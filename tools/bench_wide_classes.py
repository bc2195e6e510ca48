"""Inference cost of nets with many classes: VNet at C in {2, 16, 17, 32, 64, 127}, modes fp16 and fp32x, one JSON line per
(C, mode) plus a first line with the card's name and power limit read in the same run.

    python tools/bench_wide_classes.py [--classes 2,16,17,32,64,127] [--modes fp16,fp32x] [--reps 5] [--out DIR]

Per line: forward ms per batch of 36 x 96^3; out_block.conv1 and each tail launch in ms (CUDA events around every launch,
averaged over --reps profiled forwards after a warm-up); the tail's achieved GB/s from the bytes its plan entry computes
from shapes, and its share of the HBM bound (bytes / 7.7 TB/s over the measured time); sliding-window Mvox/s over a
512 x 512 x 400 volume (96^3 patches, stride 96, 36 per forward, volume already on the device); peak device memory of the
run; at C = 32 the time of pick_largest_cc (seg3d_cc_filter over labels 1..31) on the resulting mask.
Results: profiles/r03_wide_classes.md."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

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


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def one(C, mode, reps, B=36, S=96):
    from oracle import init as oinit
    from segmentation3d._b200.plan import NetPlan
    from segmentation3d.core.seg_infer import _cc_filter_device, make_model, segmentation_volume_device
    from segmentation3d.network.vnet import SegmentationNet
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, C, 0), 5)
    rec = {'classes': C, 'mode': mode, 'batch': '%dx%d^3' % (B, S)}
    p = NetPlan(sd, mode=mode, device='cuda')
    x = torch.randn((B, 1, S, S, S), generator=torch.Generator(device='cuda').manual_seed(1), device='cuda')
    ws, ops = p.plan(B, S, S, S)
    p.load_input(ws, x)
    for _ in range(2):
        p.run(ws, ops)
    torch.cuda.synchronize()
    rec['forward_ms'] = round(events_ms(lambda: p.run(ws, ops), reps), 3)
    prof = {}
    for _ in range(reps):
        for m, ms in p.run_profiled(ws, ops):
            prof.setdefault(m['name'], [m, 0.0])[1] += ms / reps
    c1 = prof['out_block.conv1']
    rec['conv1_ms'] = round(c1[1], 3)
    rec['conv1_kind'] = c1[0]['kind']
    rec['conv1_cout'] = p.convs['out_block.conv1'].cout
    for name, key in (('out_block.tail_stats', 'tail_stats'), ('out_block.tail_probs', 'tail_probs')):
        m, ms = prof[name]
        rec[key + '_ms'] = round(ms, 3)
        rec[key + '_kind'] = m['kind']
        rec[key + '_GBps'] = round(m['bytes'] / (ms * 1e-3) / 1e9, 1)
        rec[key + '_hbm_share'] = round(m['bytes'] / HBM_BPS / (ms * 1e-3), 3)
    del ws, ops, x
    p._plans.clear()
    # sliding window over the benchmark volume
    net = SegmentationNet(1, C)
    net.load_state_dict(sd)
    net.b200_mode = mode
    net = net.cuda().eval()
    model = make_model(net, [1.0, 1.0, 1.0], None, batch=B)
    Z, Y, X = 400, 512, 512
    vol = torch.randn((Z, Y, X), generator=torch.Generator(device='cuda').manual_seed(2), device='cuda')
    cfg = {'partition_type': 'SIZE', 'partition_size': [S, S, S], 'partition_stride': [S, S, S]}
    with torch.no_grad():
        acc, mask = segmentation_volume_device(model, cfg, vol, batch=B)
        del acc, mask
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        acc, mask = segmentation_volume_device(model, cfg, vol, batch=B)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    rec['sliding_Mvox_s'] = round(Z * Y * X / dt / 1e6, 1)
    if C == 32:
        _cc_filter_device(mask, list(range(1, C)), 0)
        torch.cuda.synchronize()
        rec['pick_largest_cc_ms'] = round(events_ms(lambda: _cc_filter_device(mask, list(range(1, C)), 0), 3), 2)
    rec['peak_mem_GB'] = round(torch.cuda.max_memory_allocated() / 1e9, 1)
    del acc, mask, vol, model, net, p
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--classes', default='2,16,17,32,64,127')
    ap.add_argument('--modes', default='fp16,fp32x')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None, help='also append the lines to DIR/bench_wide_classes.jsonl')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_wide_classes: needs a CUDA device')
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    for C in [int(c) for c in a.classes.split(',')]:
        for mode in a.modes.split(','):
            rec = one(C, mode, a.reps)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'bench_wide_classes.jsonl'), 'a') as f:
            for r in lines:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
