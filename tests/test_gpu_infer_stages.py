"""Every launch of the inference forward (segmentation3d/_b200/plan.py, one pass, no CUDA graph) against a float64
recomputation from the very buffers that launch read, up to the benchmarked 36-patch batch of 96^3.

The ops of the plan are issued one at a time (ops[i] is described by ws['meta'][i]); after each launch its output is held to

    |got - ref| <= rel |ref| + frac mag + abs

with `mag` the float64 value of the same expression with every term replaced by its magnitude, `rel` half an ulp of the
stored type (2^-11 fp16, 2^-24 fp32), `abs` half the smallest fp16 subnormal (2^-25) for fp16 stores, and `frac` from the
kernel's own fp32 accumulation: (S + 2) 2^-23 for a tensor-core convolution whose accumulator takes S MMA K-steps (a
truncating accumulator may lose one ulp per step), 27 2^-24 for the CUDA-core input block of the strict mode.  Weights
are the parameters rounded to the packed type (fp32x: whi + wlo; the split convolution is conv(hi + lo, whi) +
conv(hi, wlo), the three products the kernels sum).  The GroupNorm sums a producer adds are held to the storage rounding
of the tensor they are checked against plus the fp32 partial one thread forms before its flush, counted from the launch
geometry (stats_terms).  Every activation and scratch buffer starts as NaN, so an unwritten voxel fails, and every element
of a destination outside the launch's output window must keep its bits.
"""
import importlib
import math
import time

import pytest
import torch

from oracle import init as oinit
from f64_stage_ref import EPS32, _affine32, _close, _mean_rstd32, _rows, _window, conv_forward  # noqa: F401

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                   # unit roundoff of fp32
F16_REL, F16_ABS = 2.0 ** -11, 2.0 ** -25

# arch, classes, mode, B, D, H, W
CASES = [('vnet', 2, 'fp16', 36, 96, 96, 96),       # the benchmark forward (bench.py --batch 36), bench input
         ('vbnet', 5, 'fp32x', 36, 96, 96, 96),     # mode='auto' of a multi-class net (bench.py --arch vbnet --classes 5)
         ('vnet', 2, 'fp16', 2, 32, 32, 32),        # z-march with nseg > 1
         ('vbnet', 5, 'fp16', 3, 16, 32, 48),       # bottleneck units, narrow fold at 5 classes, odd batch, level-4 dims 1x2x3
         ('vnet', 9, 'fp16', 2, 32, 32, 32)]        # out_block.conv1 padded to 16 on the generic kernel, fp32 rows of pitch 9
BENCH = CASES[0]


def _sms():
    try:
        return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    except (RuntimeError, AssertionError):           # the CPU dry run (tests/dryrun_gpu_tests_on_cpu.py): a B200's count
        return 148


def _cdiv(a, b):
    return -(-a // b)


def _c1024(v):
    return (v + 1023) & ~1023


# ---- launch geometry (csrc/conv_tc.cu, conv_tc_narrow.cu, conv_tc_cin1t.cu, conv_simt.cu, elementwise.cu) -----------
def _zsegments(N, D, cols_per_sample, want, grid_cap):
    """z segments of the z-marching kernels: (lseg, items of one sample that one CTA takes, at most)"""
    cols = N * cols_per_sample
    nseg = max(1, _cdiv(want, cols))
    lseg = _cdiv(D, nseg)
    if lseg < 8:
        lseg = min(D, 8)
    nseg = _cdiv(D, lseg)
    grid = min(cols * nseg, grid_cap)
    return lseg, _cdiv(cols_per_sample * nseg, grid)


def zmarch_geometry(N, D, H, W, KC, Cout):
    """conv3d_k3_zmarch_kernel: (lseg, items per sample per CTA) as seg3d_conv_tc picks them"""
    sms = _sms()
    row = 2 * KC
    ring = (200 * 1024 // 2 - 27 * _c1024(Cout * row)) // _c1024(180 * row)
    ctas = 2 if ring >= 3 else 1
    return _zsegments(N, D, (W // 8) * _cdiv(H, 16), 4 * ctas * sms, ctas * sms)


def tc_tiles(mode, Cin, Cout, D, H, W):
    """conv3d_tc_persistent_kernel: (tiles per sample, GEMM N of a tile, CTAs per SM)"""
    from segmentation3d._b200 import lib
    conv = 1 if mode == lib.CONV_K2S2 else (2 if mode == lib.CONV_T2S2 else 0)
    Do, Ho, Wo = (D // 2, H // 2, W // 2) if conv == 1 else (D, H, W)
    npass, n = 1, Cout
    if conv == 2:
        n = min(8 * Cout, 256)
        npass = 8 * Cout // n
    KC = 64 if Cin % 64 == 0 else (32 if Cin % 32 == 0 else 16)
    slab = _c1024(n * 2 * KC)
    kwfuse = conv == 0 and Wo % 8 == 0 and 10 * 16 * 2 * KC + 3 * slab <= 48 * 1024
    best, tiles = None, None
    tw = 8 if kwfuse else 1
    while tw <= (8 if kwfuse else 32):
        th = 1
        while th <= 128 // tw:
            td = 128 // (tw * th)
            t = _cdiv(Wo, tw) * _cdiv(Ho, th) * _cdiv(Do, td)
            sc = t * 1024 - tw * 8 - th + (512 if (tw > 16 or th > 16 or td > 16) else 0)
            if best is None or sc < best:
                best, tiles = sc, t
            th *= 2
        tw *= 2
    acc = 16 if n <= 16 else (32 if n <= 32 else (64 if n <= 64 else (128 if n <= 128 else 256)))
    return tiles * npass, n, min(2, 512 // (2 * acc))


def conv_path(plan, name, x, y, D, W, meta):
    """which kernel seg3d_conv3d_fwd / _split_fwd runs for this launch"""
    from segmentation3d._b200 import lib
    c = plan.convs[name]
    if meta['kind'] == 'conv_tc_cin1':
        return 'cin1t'
    if meta['kind'] == 'conv_tc_narrow':
        return 'narrow'
    if c.impl == lib.IMPL_SIMT:
        return 'simt'
    if c.mode == lib.CONV_K3 and W % 8 == 0 and D >= 4:
        if plan.split:
            if c.cin in (16, 32) and x.ld // 2 == c.cin and y.ld % 4 == 0:
                return 'zmarch'
        elif c.cin in (16, 32, 64):
            return 'zmarch'
    return 'persistent'


def mma_steps(plan, name, path):
    """S: MMA K-steps (of K = 16) one tensor-memory accumulator takes for one output; fp32 adds for the others"""
    from segmentation3d._b200 import lib
    c = plan.convs[name]
    k = 3 if plan.split else 1                           # hi*whi, lo*whi, hi*wlo
    if path == 'cin1t':
        return 9                                         # one K = 16 step per (kd, kh) Toeplitz slab
    if path == 'narrow':
        return 3 * c.cin // 16 * k + 9                   # three kd taps in tensor memory, nine in-plane taps added in fp32
    taps = {lib.CONV_K3: 27, lib.CONV_K2S2: 8, lib.CONV_T2S2: 1}[c.mode]
    return taps * _cdiv(c.cin, 16) * k


def stats_terms(plan, name, path, N, dims_in, dims_out, cout):
    """values one epilogue thread adds into its fp32 partial GroupNorm sums before the flush, plus the float steps of the
    warp / block reduction behind it"""
    from segmentation3d._b200 import lib
    D, H, W = dims_in
    sms = _sms()
    c = plan.convs[name] if name in plan.convs else None
    if path == 'zmarch':
        kc = c.cin * (2 if plan.split else 1)
        lseg, k = zmarch_geometry(N, D, H, W, kc, c.cout)
        return k * lseg * 16 * _cdiv(c.cout, 32) + 5
    if path == 'persistent':
        tiles, n, ctas = tc_tiles(c.mode, c.cin, c.cout, D, H, W)
        grid = min(tiles * N, ctas * sms)
        return _cdiv(tiles, grid) * 16 * _cdiv(n, 32) + 5
    if path == 'narrow':                                  # CTAs per SM 1..4 depending on shared memory: take the worst
        worst = 0
        for ctas in (1, 2, 4):
            lseg, k = _zsegments(N, D, (W // 8) * _cdiv(H, 10), 4 * ctas * sms, ctas * sms)
            worst = max(worst, k * lseg * cout)
        return worst + 5
    if path == 'cin1t':                                   # per-channel sums of 4 voxels per plane, 16 channels at the flush
        lseg, k = _zsegments(N, D, _cdiv(W, 32) * _cdiv(H, 32), 8 * sms, sms)
        return k * lseg * 4 + 16 + 2 + 5
    if path == 'simt':                                    # one block: 8 voxels x <= 4 columns (16 for the input block)
        return 16 + 8 + 1 if c.cin == 1 else 32 + 8 + 1
    if path == 'tail':
        nvox = dims_out[0] * dims_out[1] * dims_out[2]
        gx = min(max(1, _cdiv(nvox, 256)), 4 * sms)
        return _cdiv(nvox, gx * 256) * cout + 8 + 1
    raise AssertionError(path)


# ---- the run --------------------------------------------------------------------------------------------------------
def _bench_input(plan, ws, B, P):
    """the first z layer of the benchmark volume's 96^3 patch grid, cropped and normalised by the gather kernel exactly as
    SlidingWindow.accumulate feeds the plan"""
    import numpy as np
    import bench
    from segmentation3d._b200 import lib
    X, Y, Z = 512, 512, 400
    vol = bench.synth_ct([X, Y, Z], 1234).cuda()
    xs = sorted(set(list(range(0, X - P, P)) + [X - P]))
    ys = sorted(set(list(range(0, Y - P, P)) + [Y - P]))
    starts = [[x, y, 0] for y in ys for x in xs]
    assert len(starts) == B
    sd = torch.tensor(np.asarray(starts, dtype=np.int32), dtype=torch.int32).cuda()
    nm = bench.NORMALIZER
    args = (lib.ptr(vol), Z, Y, X, lib.ptr(sd), B, P, P, P, lib.NORM_FIXED, float(nm['mean']), float(nm['stddev']),
            1 if nm['clip'] else 0, -1.0, 1.0, None, plan.in_dt)
    if ws.get('x_pad'):
        lib.call('seg3d_patch_gather_rows', *args, lib.ptr(ws['x_in']), P + lib.CIN1_PAD, lib.CIN1_LEFT, lib.stream_ptr())
    else:
        lib.call('seg3d_patch_gather', *args, lib.ptr(ws['x_in']), lib.stream_ptr())
    torch.cuda.synchronize()


def _nan_fill(ws):
    for k, v in ws.items():
        if k[:3] in ('cat', 'raw') or k[:1] in 'ATUM' or k == 'probs':
            if isinstance(v, torch.Tensor):
                v.fill_(float('nan'))
    ws['tail']['raw'].buf.fill_(float('nan'))


class Run(object):
    """one inference plan with its workspaces, NaN-filled, the input loaded; launch i is issued by step(i)"""

    def __init__(self, case):
        from segmentation3d._b200 import lib
        from segmentation3d._b200.plan import NetPlan
        lib.load()
        arch, C, mode, B, D, H, W = case
        self.case, self.B = case, B
        self.sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, C, 0), 11)
        self.plan = NetPlan(self.sd, mode=mode, device=torch.zeros(1).cuda().device)
        self.plan.use_graph = False
        self.ws, self.ops = self.plan.plan(B, D, H, W)
        assert self.ws['schedule'] == [(0, len(self.ops), B)], 'one pass over the whole batch'
        assert len(self.ops) == len(self.ws['meta'])
        _nan_fill(self.ws)
        if case == BENCH or (case[3] == 36 and case[4] == 96):
            _bench_input(self.plan, self.ws, B, D)
        else:
            x = torch.randn((B, 1, D, H, W), generator=torch.Generator().manual_seed(B + D + C)).cuda()
            self.plan.load_input(self.ws, x)
        self.ws['stats'].zero_()
        self.ws['stats2'].zero_()
        self.log = {}
        self.defects = {}
        self.checked = 0

    def weight(self, name):
        """parameter rounded to the packed weight type: ([w], bias); fp32x: [whi, wlo]"""
        from segmentation3d._b200 import lib
        c = self.plan.convs[name]
        w = self.sd[name + '.weight'].detach().cuda().float()
        b = self.sd.get(name + '.bias')
        b = None if b is None else b.detach().cuda().float().double()
        if c.impl == lib.IMPL_SIMT and not c.cin1_tc:
            return [w.double()], b
        if self.plan.split:
            hi = w.half()
            return [hi.double(), (w - hi.float()).half().double()], b
        return [w.to(lib.TORCH_DTYPE[c.dt]).double()], b

    def record(self, kind, ratio):
        self.log[kind] = max(self.log.get(kind, 0.0), ratio)


def _chunks(B, per_sample_elems):
    """sample ranges whose float64 working set stays below ~6 GB"""
    k = max(1, min(B, int(6e9 // (8 * per_sample_elems))))
    return [(b0, min(k, B - b0)) for b0 in range(0, B, k)]


def _stats_row(r, gname):
    return r.ws['stats'][r.plan.gn_index[gname]]


class StatsAcc(object):
    """per-sample float64 sums of the tensor the GroupNorm sums are checked against, and of their magnitudes"""

    def __init__(self, B, dev):
        self.s, self.ss, self.m, self.mm, self.ex = [torch.zeros(B, dtype=torch.float64, device=dev) for _ in range(5)]

    def add(self, b0, nb, y, m, rel, absb, err=None):
        """y: stored values (or the float64 reference), m: |summand| the fp32 partial adds, err: bound of |y - summed|"""
        yf, mf = y.reshape(nb, -1), m.reshape(nb, -1)
        sl = slice(b0, b0 + nb)
        self.s[sl] += yf.sum(1)
        self.ss[sl] += (yf * yf).sum(1)
        self.m[sl] += mf.sum(1)
        self.mm[sl] += (mf * mf).sum(1)
        # |stored - summed| <= rel |y| + abs (+ err): the sums and the sums of squares of that difference
        e = rel * yf.abs() + absb
        if err is not None:
            e = e + err.reshape(nb, -1)
        self.ex[sl] += e.sum(1)
        self.ex2 = getattr(self, 'ex2', torch.zeros_like(self.s))
        self.ex2[sl] += (e * (2 * yf.abs() + e)).sum(1)

    def check(self, name, stats, nt):
        st = stats.double()
        tol0 = self.ex + (nt + 2) * U * self.m
        tol1 = self.ex2 + (nt + 3) * U * self.mm
        e0, e1 = (st[:, 0] - self.s).abs(), (st[:, 1] - self.ss).abs()
        ok = bool((e0 <= tol0).all()) and bool((e1 <= tol1).all())
        assert ok, '%s: GroupNorm sums out of bound: sum err %s tol %s; sum of squares err %s tol %s' % (
            name, e0.tolist()[:4], tol0.tolist()[:4], e1.tolist()[:4], tol1.tolist()[:4])
        return max(float((e0 / tol0).max()), float((e1 / tol1).max()))


def _gn_transform(r, raw, gname, b0, nb, cnt, stats=None, res=None):
    """relu(fma(raw, a, b) (+ res)) with the kernels' fp32 a, b: (value in float64 before the store, magnitude)"""
    g = r.plan.gns[gname]
    st = (_stats_row(r, gname) if stats is None else stats)[b0:b0 + nb]
    mean, rstd = _mean_rstd32(st, cnt)
    C = raw.shape[-1]
    a, b = _affine32(mean, rstd, g.gamma[:C], g.beta[:C])
    t = raw * a + b
    mag = raw.abs() * a.abs() + g.beta[:C].double().abs().view(1, 1, -1) + mean.abs() * a.abs()
    if res is not None:
        t = t + res
        mag = mag + res.abs()
    return t.clamp_min(0.0), mag, (t, a, b)


def _fl32_relu_fma(raw, a, b, res=None):
    """the fp32 value the kernels form: fl(fma(raw, a, b)) (+ res, rounded again), then ReLU"""
    t = (raw * a + b).float()
    if res is not None:
        t = (t.double() + res).float()
    return t.double().clamp_min(0.0)


# ---- per-launch checks ----------------------------------------------------------------------------------------------
def _unit_of(r, name):
    for u in r.ws['units']:
        if u['conv'] == name:
            return u
    return None


def _x_input(r, u, b0, nb, dims, xform=None):
    """the convolution input as the kernel reads it, [nb, D, H, W, C] float64 ([hi, lo] in the strict mode)"""
    from segmentation3d._b200 import lib
    D, H, W = dims
    nv = D * H * W
    x = u['x']
    if u.get('pad', False):
        xp = r.ws['x_in'].view(r.B, D, H, W + lib.CIN1_PAD)[b0:b0 + nb]
        return [xp[..., lib.CIN1_LEFT:lib.CIN1_LEFT + W].double().unsqueeze(-1)]
    if r.plan.split and x.buf.dtype != torch.float32:
        return [_rows(x, nv, b0, nb).view(nb, D, H, W, -1), _rows(_window(x, x.ld // 2, x.C), nv, b0, nb).view(nb, D, H, W, -1)]
    v = _rows(x, nv, b0, nb)
    if xform is not None:
        v = xform(v, b0, nb)
    return [v.view(nb, D, H, W, -1)]


def _conv_ref(r, name, mode, xs, ws, bias):
    """(ref, mag) of the convolution over the stored inputs: conv(hi + lo, whi) + conv(hi, wlo) in the strict mode"""
    if len(ws) == 2 and len(xs) == 2:
        hi, lo = xs
        whi, wlo = ws
        ref = conv_forward(mode, hi + lo, whi, bias) + conv_forward(mode, hi, wlo)
        mag = conv_forward(mode, hi.abs() + lo.abs(), whi.abs(), None if bias is None else bias.abs()) + conv_forward(mode, hi.abs(), wlo.abs())
        return ref, mag
    x = xs[0] if len(xs) == 1 else xs[0] + xs[1]
    w = ws[0] if len(ws) == 1 else ws[0] + ws[1]
    return conv_forward(mode, x, w, bias), conv_forward(mode, x.abs(), w.abs(), None if bias is None else bias.abs())


def check_conv(r, i, meta, u, y, gname, stats_before, xform=None, ulp_in=None, stats_override=None, y_override=None,
               cols_dropped=None):
    """one convolution launch: output window `y` (None: sums only) and the GroupNorm row it adds to"""
    from segmentation3d._b200 import lib
    plan, ws, B = r.plan, r.ws, r.B
    name = u['conv']
    c = plan.convs[name]
    din, dout = ws['dims'][u['lin']], ws['dims'][u['lout']]
    nvo = dout[0] * dout[1] * dout[2]
    path = conv_path(plan, name, u['x'], y if y is not None else u['x'], din[0], din[2], meta)
    if path == 'simt':
        frac = (27 if c.cin == 1 else 27 * c.cin) * U
    else:
        frac = (mma_steps(plan, name, path) + 2) * 2.0 ** -23
    ws_, bias = r.weight(name)
    if path == 'narrow':
        ws_ = [w[:plan.out_channels] for w in ws_]
        bias = bias[:plan.out_channels]
    else:
        ws_ = [w[:c.real_cout] if c.mode != lib.CONV_T2S2 else w[:, :c.real_cout] for w in ws_]
        bias = None if bias is None else bias[:c.real_cout]
    cout = ws_[0].shape[0] if c.mode != lib.CONV_T2S2 else ws_[0].shape[1]
    acc = StatsAcc(B, ws['stats'].device)
    worst = 0.0
    nin = din[0] * din[1] * din[2]
    for b0, nb in _chunks(B, 4 * nin * (c.cin + cout) + 2 * nvo * cout):
        xs = _x_input(r, u, b0, nb, din, xform)
        ref, mag = _conv_ref(r, name, c.mode, xs, ws_, bias)
        extra = None
        if ulp_in is not None:                          # one ulp of the storage rounding of the input formed in shared memory
            extra = F16_REL * conv_forward(c.mode, ulp_in(b0, nb).view(xs[0].shape), ws_[0].abs() if len(ws_) == 1 else ws_[0].abs() + ws_[1].abs())
            extra = extra.view(nb, nvo, -1)
        del xs
        ref, mag = ref.view(nb, nvo, -1), mag.view(nb, nvo, -1)
        if y is not None:
            got = (_rows(y, nvo, b0, nb) if y_override is None else y_override(b0, nb))
            f32 = y.buf.dtype == torch.float32
            rel, absb = (U, 0.0) if f32 else (F16_REL, F16_ABS)
            worst = max(worst, _close('%s [%d:%d]' % (name, b0, b0 + nb), got, ref, mag, rel, frac, 0.0 if f32 else absb, extra))
            acc.add(b0, nb, got, got.abs() * (1 + 2 * rel) + absb if path != 'cin1t' else mag, rel, absb)
        else:                                            # sums only: against the float64 convolution
            acc.add(b0, nb, ref, mag, 0.0, 0.0, err=frac * mag)
        del ref, mag, extra
    r.record(path if path != 'narrow' else 'narrow', worst)
    if gname is not None:
        nt = stats_terms(plan, name, path, B, din, dout, cout)
        st = _stats_row(r, gname) if stats_override is None else stats_override
        if cols_dropped is not None:
            st = cols_dropped(st)
        r.record('stats', acc.check(name + ' GroupNorm sums', st, nt))
    return acc


def check_gn_apply(r, u, out=None, stats=None):
    """seg3d_gn_apply / _split: relu(fma(raw, a, b) (+ res)), stored; strict mode: hi = fl16(t), hi + lo within 2^-22 |t|"""
    plan, ws, B = r.plan, r.ws, r.B
    nv = ws['vox'][u['lout']]
    C = u['raw'].C
    out = u['out'] if out is None else out
    split = plan.split
    worst = 0.0
    for b0, nb in _chunks(B, nv * C * 8):
        raw = _rows(u['raw'], nv, b0, nb)
        res = None
        if u['res'] is not None:
            res = _rows(u['res'], nv, b0, nb)
            if split:
                res = res + _rows(_window(u['res'], u['res'].ld // 2, C), nv, b0, nb)
        ref, mag, _ = _gn_transform(r, raw, u['gn'], b0, nb, float(nv * C), stats=stats, res=res)
        del raw, res
        got = _rows(out, nv, b0, nb)
        nm = '%s apply [%d:%d]' % (u['gn'], b0, b0 + nb)
        if split:
            lo = _rows(_window(out, out.ld // 2, C), nv, b0, nb)
            worst = max(worst, _close(nm + ' hi', got, ref, mag, F16_REL, 3 * U, F16_ABS))
            worst = max(worst, _close(nm + ' hi+lo', got + lo, ref, mag, 2.0 ** -22, 3 * U, F16_ABS))
        else:
            worst = max(worst, _close(nm, got, ref, mag, F16_REL, 2 * U, F16_ABS))
    r.record('gn_apply', worst)


def _tail_forward(r, b0, nb, stats2=None):
    """fp32 tail forward in float64 from the stored conv1 output and stats: z, |z| bound, and the GroupNorm-2 affine"""
    plan, ws = r.plan, r.ws
    nc, nv = plan.out_channels, ws['vox'][0]
    y = _rows(_window(ws['tail']['raw'], 0, nc), nv, b0, nb)
    g1, g2 = plan.gns['out_block.gn1'], plan.gns['out_block.gn2']
    m1, r1 = _mean_rstd32(_stats_row(r, 'out_block.gn1')[b0:b0 + nb], float(nv * nc))
    a1, c1 = _affine32(m1, r1, g1.gamma, g1.beta)
    h = (y * a1 + c1).clamp_min(0.0)
    habs = y.abs() * a1.abs() + c1.abs()
    W2 = plan.w2.double()
    z = h @ W2.t() + plan.b2.double().view(1, 1, nc)
    zabs = habs @ W2.abs().t() + plan.b2.double().abs().view(1, 1, nc)
    return z, zabs, (g2, stats2)


def check_tail_stats(r):
    plan, ws, B = r.plan, r.ws, r.B
    nc, nv = plan.out_channels, ws['vox'][0]
    acc = StatsAcc(B, ws['stats'].device)
    for b0, nb in _chunks(B, nv * nc * 8):
        z, zabs, _ = _tail_forward(r, b0, nb)
        acc.add(b0, nb, z, zabs, 0.0, 0.0, err=(nc + 3) * U * zabs)
    nt = stats_terms(plan, None, 'tail', B, ws['dims'][0], ws['dims'][0], nc)
    r.record('tail', acc.check('out_block.tail_stats', ws['stats2'], nt))


def check_tail_probs(r):
    """softmax(fma(z, a2, b2)) against float64; the fp32 error of each argument (z: C + 3 roundings of its magnitude, the
    FMA, the max subtraction, expf) moves p_c by p_c (e_c + sum_j p_j e_j); the division adds a few ulps"""
    plan, ws, B = r.plan, r.ws, r.B
    nc, nv = plan.out_channels, ws['vox'][0]
    worst = 0.0
    for b0, nb in _chunks(B, nv * nc * 12):
        z, zabs, (g2, _) = _tail_forward(r, b0, nb)
        m2, r2 = _mean_rstd32(ws['stats2'][b0:b0 + nb], float(nv * nc))
        a2, c2 = _affine32(m2, r2, g2.gamma, g2.beta)
        arg = z * a2 + c2
        p = torch.softmax(arg, 2)
        mx = arg.max(2, keepdim=True)[0].abs()
        e = (nc + 3) * U * a2.abs() * zabs + 2 * U * (z.abs() * a2.abs() + c2.abs() + mx) + 4 * U
        bound = p * (e + (p * e).sum(2, keepdim=True)) + 4 * U * p
        got = ws['probs'][b0:b0 + nb].double().reshape(nb, nc, nv).transpose(1, 2)
        worst = max(worst, _close('out_block.tail_probs [%d:%d]' % (b0, b0 + nb), got, p, bound, 0.0, 1.0))
    r.record('tail', worst)


# ---- destinations: nothing outside the output window may change -----------------------------------------------------
def _window_mask(buf, views, nvox, B):
    """bool mask over the flat buffer: True inside the channel windows of `views` for samples [0, B)"""
    m = torch.zeros(buf.numel(), dtype=torch.bool, device=buf.device)
    for v in views:
        base = v.off
        torch.as_strided(m, (B, nvox, v.C), (nvox * v.ld, v.ld, 1), base).fill_(True)
    return m


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else (t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int64))


def assert_outside_unchanged(name, before, after, views, nvox, B):
    changed = (_bits(before).reshape(-1) != _bits(after).reshape(-1))
    if views:
        changed &= ~_window_mask(after, views, nvox, B)
    n = int(changed.sum())
    assert n == 0, '%s: %d elements outside the output window changed' % (name, n)


# ---- walking the forward --------------------------------------------------------------------------------------------
def _describe(r, i):
    """(what launch i is, the unit it belongs to, output views, GroupNorm row it adds to or None)"""
    ws, plan = r.ws, r.plan
    m = ws['meta'][i]
    name = m['name']
    if name == 'in_block.conv.stats':
        u = dict(_unit_of(r, 'in_block.conv'), pad=True)
        return 'cin1_stats', u, [], 'in_block.gn'
    if name == 'in_block.conv.gn_relu':
        u = dict(_unit_of(r, 'in_block.conv'), pad=True)
        return 'cin1_gn_relu', u, [u['out']], None
    if name == 'out_block.conv1':
        return 'conv1', None, [ws['tail']['raw']], 'out_block.gn1'
    if name == 'out_block.tail_stats':
        return 'tail_stats', None, [], None
    if name == 'out_block.tail_probs':
        return 'tail_probs', None, [], None
    if m['kind'] == 'gn_apply':
        u = next(v for v in ws['units'] if v['gn'] == name)
        out = u['out']
        views = [out, _window(out, out.ld // 2, out.C)] if plan.split else [out]
        return 'gn_apply', u, views, None
    u = _unit_of(r, name)
    assert u is not None, name
    u = dict(u, pad=bool(u.get('xpad') is not None))
    return 'conv', u, [u['raw']], u['gn']


def _gnin(r, u):
    d = r.ws.get('deferred')
    if d is not None and d.get('res_gnin') is not None and u is not None and u['raw'] is d['raw']:
        return d['res_gnin']
    return None


def _gnin_xform(r, gn, nch, nv, stats=None):
    """the lower nch input channels are fl16(relu(fma(raw, a, b))) of GroupNorm `gn`"""
    def f(v, b0, nb):
        v = v.clone()
        _, _, (t, a, b) = _gn_transform(r, v[..., :nch], gn, b0, nb, float(nv * nch), stats=stats)
        v[..., :nch] = _fl32_relu_fma(v[..., :nch], a, b).half().double()
        return v
    return f


def check_launch(r, i, kind, u, views, gname, stats_before):
    plan, ws, B = r.plan, r.ws, r.B
    meta = ws['meta'][i]
    if kind == 'conv':
        gi = _gnin(r, u)
        if gi is None:
            check_conv(r, i, meta, u, u['raw'], gname, stats_before)
        else:                                            # seg3d_conv3d_k3_gnin_fwd
            nv = ws['vox'][u['lin']]
            xf = _gnin_xform(r, gi['gn'], gi['nch'], nv)
            ulp = lambda b0, nb: torch.cat([xf(_rows(u['x'], nv, b0, nb), b0, nb)[..., :gi['nch']].abs(),
                                            torch.zeros_like(_rows(u['x'], nv, b0, nb)[..., gi['nch']:])], -1)
            check_conv(r, i, meta, u, u['raw'], gname, stats_before, xform=xf, ulp_in=ulp)
            r.record('gnin', r.log.get('zmarch', 0.0))
    elif kind == 'gn_apply':
        check_gn_apply(r, u)
    elif kind == 'cin1_stats':
        check_conv(r, i, meta, u, None, gname, stats_before)
    elif kind == 'cin1_gn_relu':
        assert torch.equal(ws['stats'], stats_before), 'epilogue 2 of seg3d_conv3d_cin1_fwd changed the GroupNorm sums'
        u2 = dict(u, raw=None)
        check_cin1_gn_relu(r, u2)
    elif kind == 'conv1':
        check_conv1(r, i, meta, gname, stats_before)
    elif kind == 'tail_stats':
        check_tail_stats(r)
    elif kind == 'tail_probs':
        check_tail_probs(r)


def check_cin1_gn_relu(r, u):
    """epilogue 2: relu(gn(conv)) with the sums of epilogue 1; conv error propagates through a = rstd gamma"""
    plan, ws, B = r.plan, r.ws, r.B
    nv = ws['vox'][0]
    D, H, W = ws['dims'][0]
    frac = (mma_steps(plan, 'in_block.conv', 'cin1t') + 2) * 2.0 ** -23
    (w,), bias = r.weight('in_block.conv')
    worst = 0.0
    for b0, nb in _chunks(B, nv * 16 * 10):
        x = _x_input(r, u, b0, nb, (D, H, W))[0]
        y = conv_forward(plan.convs['in_block.conv'].mode, x, w, bias).view(nb, nv, 16)
        ym = conv_forward(plan.convs['in_block.conv'].mode, x.abs(), w.abs(), bias.abs()).view(nb, nv, 16)
        ref, mag, (t, a, b) = _gn_transform(r, y, 'in_block.gn', b0, nb, float(nv * 16))
        mag = mag + frac * ym * a.abs() / (2 * U)        # the convolution's own error, carried through the scale
        got = _rows(u['out'], nv, b0, nb)
        worst = max(worst, _close('in_block.conv gn_relu [%d:%d]' % (b0, b0 + nb), got, ref, mag, F16_REL, 2 * U, F16_ABS))
    r.record('cin1t', worst)


def check_conv1(r, i, meta, gname, stats_before, stats_override=None):
    """out_block.conv1: plain, narrow folded (its input formed from a deferred GroupNorm), split or padded generic"""
    plan, ws, B = r.plan, r.ws, r.B
    tail = ws['tail']
    nv = ws['vox'][0]
    u = {'conv': 'out_block.conv1', 'x': tail['x'], 'lin': 0, 'lout': 0}
    if meta['kind'] == 'conv_tc_narrow' and ws.get('deferred') is not None:
        d = ws['deferred']
        C = d['raw'].C
        rg = d.get('res_gnin')
        rxf = _gnin_xform(r, rg['gn'], rg['nch'], nv) if rg is not None else None

        def formed(b0, nb):
            res = _rows(d['res'], nv, b0, nb)
            if rxf is not None:
                res = rxf(res, b0, nb)
            raw = _rows(d['raw'], nv, b0, nb)
            _, _, (t, a, b) = _gn_transform(r, raw, d['gn'], b0, nb, float(nv * C))
            return _fl32_relu_fma(raw, a, b, res).half().double()
        u = dict(u, x=d['raw'])
        check_conv(r, i, meta, u, tail['raw'], gname, stats_before, xform=lambda v, b0, nb: formed(b0, nb),
                   ulp_in=lambda b0, nb: formed(b0, nb).abs(), stats_override=stats_override)
        r.record('narrow_gn2' if rg is not None else 'narrow_gn', r.log.get('narrow', 0.0))
    else:
        check_conv(r, i, meta, u, tail['raw'], gname, stats_before, stats_override=stats_override)


def walk(case, probe=None):
    """issue every launch of the forward once, checking each against float64 right after it ran"""
    r = Run(case)
    ws, ops, B = r.ws, r.ops, r.B
    t0 = time.time()
    for i, op in enumerate(ops):
        kind, u, views, gname = _describe(r, i)
        if gname is not None:
            row = _stats_row(r, gname)
            assert bool((row == 0).all()), '%s: GroupNorm row not zero before its producer' % ws['meta'][i]['name']
        dests = list({id(v.buf): v.buf for v in views}.values())     # tail_probs: the whole of `probs` is its output
        before = [d.clone() for d in dests]
        stats_before = ws['stats'].clone()
        stats2_before = ws['stats2'].clone()
        op(0, B)
        torch.cuda.synchronize()
        for d, b in zip(dests, before):
            nvox = ws['vox'][u['lout']] if u is not None else ws['vox'][0]
            vs = [v for v in views if v.buf is d]
            assert_outside_unchanged(ws['meta'][i]['name'], b, d, vs, nvox, B)
        del before
        # only the launch's own GroupNorm row (or stats2 for the tail) may change
        keep = torch.ones(ws['stats'].shape[0], dtype=torch.bool, device=ws['stats'].device)
        if gname is not None and kind != 'cin1_gn_relu':
            keep[r.plan.gn_index[gname]] = False
        assert torch.equal(ws['stats'][keep], stats_before[keep]), '%s wrote another GroupNorm row' % ws['meta'][i]['name']
        if kind != 'tail_stats':
            assert torch.equal(ws['stats2'], stats2_before), '%s wrote stats2' % ws['meta'][i]['name']
        check_launch(r, i, kind, u, views, gname, stats_before)
        if probe is not None:
            probe(r, i, kind, u, views, gname)
        r.checked += 1
    torch.cuda.synchronize()
    r.seconds = time.time() - t0
    return r


def _report(r):
    print('%s: %d launches checked against float64 (plan.launches = %d), %.0f s' % (str(r.case), r.checked, r.plan.launches(r.ws), r.seconds))
    try:
        print('    peak device memory %.1f GB' % (torch.cuda.max_memory_allocated() / 1e9))
    except (RuntimeError, AssertionError):
        pass
    for k in sorted(r.log):
        print('    %-12s worst err / bound %.3f' % (k, r.log[k]))


# ---- the bench forward, and the checks can fail ---------------------------------------------------------------------
DEFECTS = ['zmarch_last_plane_zeroed', 'gn_stats_samples_swapped', 'stats_column_dropped', 'gnin_next_sample_stats',
           'gn_apply_voxel_nan']
_BENCH = {}


def _rejects(fn):
    try:
        fn()
    except AssertionError:
        return True
    return False


def _bench_probe(r, i, kind, u, views, gname):
    """perturbed copies of the launch's real buffers through the same checks; the real ones passed just before"""
    ws, B = r.ws, r.B
    D, H, W = ws['dims'][0]
    nv = D * H * W
    meta = ws['meta'][i]
    if kind == 'conv' and _gnin(r, u) is not None:           # up_32.rblock.ops.0.conv: a level-0 z-march with the transform
        gi = _gnin(r, u)
        y = u['raw']

        def zeroed(b0, nb):
            g = _rows(y, nv, b0, nb)
            if b0 + nb == B:
                g.view(nb, D, H * W, -1)[-1, D - 1] = 0
            return g
        xf = _gnin_xform(r, gi['gn'], gi['nch'], nv)
        ulp = lambda b0, nb: xf(_rows(u['x'], nv, b0, nb), b0, nb).abs()
        r.defects['zmarch_last_plane_zeroed'] = _rejects(lambda: check_conv(r, i, meta, u, y, None, None, xform=xf, ulp_in=ulp, y_override=zeroed))
        # one 8 x 16 column (all D planes) of the last sample taken out of the sums
        g = _rows(y, nv, B - 1, 1).view(D, H, W, -1)[:, :16, :8]
        col = torch.tensor([float(g.sum()), float((g * g).sum())], dtype=torch.float64, device=g.device)

        def drop(st):
            st = st.clone()
            st[B - 1] -= col
            return st
        r.defects['stats_column_dropped'] = _rejects(lambda: check_conv(r, i, meta, u, y, gname, None, xform=xf, ulp_in=ulp,
                                                                        cols_dropped=drop))
        # the transform formed with the next sample's GroupNorm statistics
        upst = _stats_row(r, gi['gn'])
        shifted = torch.roll(upst, -1, 0)
        xbad = _gnin_xform(r, gi['gn'], gi['nch'], nv, stats=shifted)
        r.defects['gnin_next_sample_stats'] = _rejects(lambda: check_conv(r, i, meta, u, y, None, None, xform=xbad, ulp_in=ulp))
    if kind == 'gn_apply' and 'gn_stats_samples_swapped' not in r.defects:
        st = _stats_row(r, u['gn']).clone()
        st[[0, B - 1]] = st[[B - 1, 0]]
        r.defects['gn_stats_samples_swapped'] = _rejects(lambda: check_gn_apply(r, u, stats=st))
        out = u['out']
        bad = out.buf.clone()
        from segmentation3d._b200.plan import _View
        bv = _View(bad, out.off, out.ld, out.C)
        flat = bad.view(-1)
        nvu = ws['vox'][u['lout']]
        flat[out.off + ((B - 1) * nvu + nvu // 2) * out.ld + out.C - 1] = float('nan')
        r.defects['gn_apply_voxel_nan'] = _rejects(lambda: check_gn_apply(r, u, out=bv))


def _bench_run():
    if 'r' not in _BENCH:
        _BENCH['r'] = walk(BENCH, probe=_bench_probe)
    return _BENCH['r']


_ID = lambda c: '%s%d-%s-%dx%dx%dx%d' % c


@pytest.mark.parametrize('case', CASES, ids=_ID)
def test_every_inference_launch_matches_float64(case):
    r = _bench_run() if case == BENCH else walk(case)
    _report(r)
    assert r.checked == r.plan.launches(r.ws) == len(r.ops)


@pytest.mark.parametrize('case', [BENCH], ids=_ID)
def test_infer_stage_checks_reject_injected_defects(case):
    """on the 36 x 96^3 run: a zeroed last z-plane of the last sample of a level-0 z-march output; two samples' GroupNorm rows
    swapped before a gn_apply check; one 8 x 16 column (all 96 planes) of one sample taken out of a level-0 conv's sums; the
    gnin transform formed with the next sample's statistics; one voxel of a gn_apply output set back to NaN"""
    r = _bench_run()
    print('defects rejected: %s' % r.defects)
    assert sorted(r.defects) == sorted(DEFECTS), r.defects
    assert all(r.defects.values()), r.defects
