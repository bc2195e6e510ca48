"""Time conv3d_k3_zmarch_kernel at the benchmark's level-0/1 shapes under different residency / plane-ring settings:
two CTAs per SM with a 3-plane ring each (the default for 32->32) against one CTA per SM with 4 to 11 planes.

The launcher reads SEG3D_ZM_CTAS_PER_SM and SEG3D_ZM_RING on every call, so the settings alternate inside one process:
every round times every setting once per case.  Inputs rotate over three buffers (6 GB at 96^3, 0.8 GB at 48^3, both larger
than the 126 MB L2); CUDA events around `reps` launches.  The z-segment length is pinned to what the two-CTA default
picks, so the settings differ only in CTAs per SM and plane-ring depth.

usage: python tools/zmarch_ring_sweep.py [--rounds 3] [--reps 20] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'medical-segmentation3d-toolkit_b200'))
import torch
from segmentation3d._b200 import lib as L

SETTINGS = [('2cta_ring3', {'SEG3D_ZM_CTAS_PER_SM': '2', 'SEG3D_ZM_RING': '3'}),
            ('1cta_ring4', {'SEG3D_ZM_CTAS_PER_SM': '1', 'SEG3D_ZM_RING': '4'}),
            ('1cta_ring6', {'SEG3D_ZM_CTAS_PER_SM': '1', 'SEG3D_ZM_RING': '6'}),
            ('1cta_ring8', {'SEG3D_ZM_CTAS_PER_SM': '1', 'SEG3D_ZM_RING': '8'}),
            ('1cta_ring11', {'SEG3D_ZM_CTAS_PER_SM': '1', 'SEG3D_ZM_RING': '11'})]
# (name, N, D, xf): 32->32 plain at levels 0 and 1, and the XF form up_32.rblock.ops.0.conv runs in the benchmark
CASES = [('32x32@96', 36, 96, False), ('32x32@48', 36, 48, False), ('32x32xf@96', 36, 96, True)]


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def default_lseg(N, D, H, W):
    """the z-segment length seg3d_conv_tc picks for 32->32 at two CTAs per SM"""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cols = N * (W // 8) * -(-H // 16)
    nseg = max(1, -(-4 * 2 * sms // cols))
    lseg = -(-D // nseg)
    return min(D, 8) if lseg < 8 else lseg


class Case:
    def __init__(self, N, D, xf, cin=32, cout=32):
        g = torch.Generator(device='cuda').manual_seed(1)
        self.N, self.D, self.xf, self.cin, self.cout = N, D, xf, cin, cout
        self.x = [torch.randn((N, D, D, D, cin), device='cuda', generator=g).half() for _ in range(3)]
        self.w = (torch.randn((27, cout, cin), device='cuda', generator=g) * 0.05).half()
        self.b = torch.randn(cout, device='cuda', generator=g) * 0.1
        self.y = torch.empty((N, D, D, D, cout), device='cuda', dtype=torch.half)
        self.stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
        cnt = 16.0 * D ** 3                                 # transformed half: GroupNorm(1, 16) sums with mean 0, variance 1
        self.xf_stats = torch.tensor([[0.0, cnt]] * N, dtype=torch.float64, device='cuda')
        self.gamma = torch.ones(16, device='cuda')
        self.beta = torch.zeros(16, device='cuda')
        self.lseg = default_lseg(N, D, D, D)

    def go(self, i):
        N, D, cin, cout = self.N, self.D, self.cin, self.cout
        if self.xf:
            L.call('seg3d_conv3d_k3_gnin_fwd', L.F16, L.ptr(self.x[i % 3]), cin, cin, 16, L.ptr(self.xf_stats), L.ptr(self.gamma),
                   L.ptr(self.beta), 1e-5, L.ptr(self.w), L.ptr(self.b), L.ptr(self.y), cout, cout, N, D, D, D, L.ptr(self.stats),
                   L.stream_ptr())
        else:
            L.call('seg3d_conv3d_fwd', L.CONV_K3, L.F16, L.IMPL_TCGEN05, L.ptr(self.x[i % 3]), cin, cin, L.ptr(self.w), L.ptr(self.b),
                   L.ptr(self.y), cout, cout, N, D, D, D, L.ptr(self.stats), L.stream_ptr())

    def time(self, reps):
        for i in range(3):
            self.go(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            self.go(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def tflops(self, ms):
        return 2.0 * self.N * self.D ** 3 * 27 * self.cin * self.cout / ms / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    L.load()
    dev = card()
    print('card: %s' % dev, flush=True)
    cases = [(name, Case(N, D, xf)) for name, N, D, xf in CASES]
    res = {name: {s: [] for s, _ in SETTINGS} for name, _ in cases}
    for r in range(a.rounds):
        for name, c in cases:
            for s, env in SETTINGS:
                os.environ.update(env)
                os.environ['SEG3D_ZM_LSEG'] = str(c.lseg)
                ms = c.time(a.reps)
                res[name][s].append(ms)
                print('round %d %-11s %-12s %.4f ms %6.0f TFLOP/s' % (r, name, s, ms, c.tflops(ms)), flush=True)
    for k in ('SEG3D_ZM_CTAS_PER_SM', 'SEG3D_ZM_RING', 'SEG3D_ZM_LSEG'):
        os.environ.pop(k, None)
    print('\nmedian over %d rounds (ms, TFLOP/s, vs 2cta_ring3):' % a.rounds)
    summary = {}
    for name, c in cases:
        base = sorted(res[name]['2cta_ring3'])[a.rounds // 2]
        for s, _ in SETTINGS:
            v = sorted(res[name][s])
            med = v[a.rounds // 2]
            summary.setdefault(name, {})[s] = {'ms': v, 'median_ms': med, 'tflops': c.tflops(med)}
            print('%-11s %-12s %.4f ms  [%.4f..%.4f]  %6.0f TFLOP/s  %+.1f %%' % (name, s, med, v[0], v[-1], c.tflops(med),
                                                                                100.0 * (base / med - 1)))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump({'card': dev, 'lseg': {n: c.lseg for n, c in cases}, 'results': summary}, f, indent=1)


if __name__ == '__main__':
    main()
