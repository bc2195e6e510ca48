"""Every stage of the bf16 training backward (segmentation3d/_b200/autograd.py::_Backward.run) against a float64
recomputation from the very tensors that stage's kernel read, up to the benchmarked VNet step (8 x 96^3, MultiDice).

An end-to-end comparison of the bf16 gradients cannot be tight (tests/test_gpu_train.py::test_bf16_training_gradients:
the rounded program is ill-conditioned below level 2).  Stage by stage nothing is amplified: the inputs of a stage are
the stored bf16 / fp32 buffers of the real run (exact in float64), so each output is held to its own rounding:

  * bf16 outputs (gy, dres, gd, gy_tail, gd_tail):  |got - ref| <= 2^-8 |ref| + 1e-5 mag      (half an ulp of bf16)
  * fp32 parameter gradients:                       |got - ref| <= 2e-5 mag                    (fp32 accumulation)
  * conv weight gradients:                         |got - ref| <= max(2e-5, (S + P) 2^-23) mag  (see wgrad_bound)

where `mag` is the float64 value of the same expression with every term replaced by its magnitude (for a convolution
conv(|gy|, |w|), for a weight gradient sum |x| |gy|).  The upstream gradient of each unit is derived here from the
channel spans of the workspace views, not from the backward's own wiring, and the ReLU masks are the kernels' own:
the stored `out > 0` where a residual is added, else the sign of fma(y, a, b) with a = fl(rstd * gamma) and
b = fl(beta - mean * a) (one rounding: the kernels form it with an FFMA), which float64 evaluates exactly.
"""
import importlib

import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from f64_stage_ref import EPS32, _affine32, _close, _mean_rstd32, _rows, _taps, _window  # noqa: F401

pytestmark = pytest.mark.gpu

BF16_REL = 2.0 ** -8        # half an ulp of bf16 (8 significant bits)
BF16_MAG = 1e-5             # fp32 arithmetic in front of the bf16 store
F32_MAG = 2e-5              # fp32 accumulation of a parameter gradient, relative to the sum of magnitudes

# arch, classes, loss, B, D, H, W
CASES = [('vnet', 2, 'dice', 2, 32, 32, 32),
         ('vbnet', 5, 'focal', 3, 16, 32, 48),        # bottleneck units, padded tail, odd batch, level-4 dims 1 x 2 x 3
         ('vnet', 16, 'ce', 2, 32, 32, 32),           # widest tail, no padding
         ('vnet', 2, 'dice', 8, 96, 96, 96)]          # BASELINE configs[2], as bench.py --task train runs it (last: the
BENCH = CASES[-1]                                     # defect tests below reuse its run)

# consumers of every VNet unit's output: a skip tensor feeds the next down conv and, through the concat buffer, the up
# block's first conv and its residual; a block input feeds its first conv and the last conv's residual
VNET_CONSUMERS = {
    'in_block.conv': 3,
    'down_32.down_conv': 2, 'down_32.rblock.ops.0.conv': 3,
    'down_64.down_conv': 2, 'down_64.rblock.ops.0.conv': 1, 'down_64.rblock.ops.1.conv': 3,
    'down_128.down_conv': 2, 'down_128.rblock.ops.0.conv': 1, 'down_128.rblock.ops.1.conv': 1, 'down_128.rblock.ops.2.conv': 3,
    'down_256.down_conv': 2, 'down_256.rblock.ops.0.conv': 1, 'down_256.rblock.ops.1.conv': 1, 'down_256.rblock.ops.2.conv': 1,
    'up_256.up_conv': 2, 'up_256.rblock.ops.0.conv': 1, 'up_256.rblock.ops.1.conv': 1, 'up_256.rblock.ops.2.conv': 1,
    'up_128.up_conv': 2, 'up_128.rblock.ops.0.conv': 1, 'up_128.rblock.ops.1.conv': 1, 'up_128.rblock.ops.2.conv': 1,
    'up_64.up_conv': 2, 'up_64.rblock.ops.0.conv': 1, 'up_64.rblock.ops.1.conv': 1,
    'up_32.up_conv': 2, 'up_32.rblock.ops.0.conv': 1,
}


# ---- comparison helpers ---------------------------------------------------------------------------------------------
def check_bf16(name, got, ref, mag):
    _close(name, got, ref, mag, BF16_REL, BF16_MAG)


def check_f32(name, got, ref, mag):
    _close(name, got, ref, mag, 0.0, F32_MAG)


def check_wgrad(name, got, ref, mag, frac):
    _close(name, got, ref, mag, 0.0, frac)


def _num_sms():
    try:
        return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    except (RuntimeError, AssertionError):           # the CPU dry run (tests/dryrun_gpu_tests_on_cpu.py): a B200's count
        return 148


def _cdiv(a, b):
    return -(-a // b)


def wgrad_steps(r, u):
    """(S, P) of the seg3d_conv3d_wgrad path that runs for unit u, from that path's launch geometry (csrc/backward.cu,
    wgrad_tc9.cu, conv_tc.cu, conv_tc_cin1t.cu): S = sequential fp32 steps into one accumulator (MMA K-steps of the tiles one
    CTA sums in tensor memory, or fmaf steps of a CUDA-core chunk), P = partial sums added per weight by atomics"""
    from segmentation3d._b200 import lib
    ws, plan = r['ws'], r['plan']
    c = plan.convs[u['conv']]
    B, sms = ws['B'], _num_sms()
    D, H, W = ws['dims'][u['lin']]
    cin, cout, x_ld, dy_ld = c.cin, c.cout, u['x'].ld, c.cout
    if u.get('xpad') is not None and cout == 16:          # input block: Toeplitz operands, one tensor-memory sum per CTA
        cols = B * _cdiv(W, 32) * _cdiv(H, 32)
        nseg = max(1, _cdiv(6 * sms, cols))
        lseg = _cdiv(D, nseg)
        if lseg < 8:
            lseg = min(D, 8)
        nitems = cols * _cdiv(D, lseg)
        grid = min(nitems, sms)
        return _cdiv(nitems, grid) * lseg * 8, grid + 8
    nblk = 64 if cin >= 64 else cin
    mblk = 128 if cout >= 128 else cout
    tc = (cin % 16 == 0 and cout % 16 == 0 and x_ld % 8 == 0 and dy_ld % 8 == 0 and cin % nblk == 0 and nblk in (16, 32, 64)
          and cout % mblk == 0)
    if tc:
        if c.mode == lib.CONV_K3:
            ntiles = _cdiv(W, 8) * _cdiv(H, 16) * D * B
            if cout in (16, 32):                          # nine taps per MMA
                combos = cin // nblk * 3
            else:
                combos = cout // mblk * (cin // nblk) * (27 // (9 if nblk <= 32 else 3))
        else:                                             # stride-2 / transposed: tiles of the low-resolution grid
            Dl, Hl, Wl = (D // 2, H // 2, W // 2) if c.mode == lib.CONV_K2S2 else (D, H, W)
            ntiles = _cdiv(Wl, 8) * _cdiv(Hl, 16) * Dl * B
            combos = cout // mblk * (cin // nblk) * 4
        ksplit = min(max(1, sms // combos), ntiles)      # one wave: every CTA sums ntiles / ksplit tiles of 8 K-steps
        return _cdiv(ntiles, ksplit) * 8, ksplit
    taps = 27 if c.mode == lib.CONV_K3 else 8            # CUDA cores: chunks of >= 512 voxels per CTA
    vps = (D // 2) * (H // 2) * (W // 2) if c.mode == lib.CONV_K2S2 else D * H * W
    want = max(1, _cdiv(4 * sms, taps * _cdiv(cin, 64) * _cdiv(cout, 64) * B))
    chunk = _cdiv(vps, want)
    if chunk < 512:
        chunk = min(vps, 512)
    chunk = _cdiv(chunk, 16) * 16
    return chunk, B * _cdiv(vps, chunk)


def wgrad_bound(r, u):
    """Bound of a weight gradient relative to sum |x| |dy|.  A tensor-core fp32 accumulator truncates instead of rounding to
    nearest, so each of its S steps may lose up to one ulp (2^-23) of the running sum, which is at most sum |x| |dy|; the P
    partial sums then go through fp32 atomics (at most half an ulp each, counted as one).  Worst case: (S + P) 2^-23, never
    below the 2e-5 of an fp32 sum (test_conv_wgrad_matches_torch).  Small shapes stay at 2e-5; one wave over 8 x 96^3 puts
    ~1 100 tiles into one CTA at level 0 and the bound reaches ~1e-3 (test_bench_step_weight_gradients_meet_the_fp32_bound)."""
    S, P = wgrad_steps(r, u)
    return max(F32_MAG, (S + P) * 2.0 ** -23)


def gn_reference(gs, y, stats, gamma, beta, out=None):
    """GroupNorm(1, C) + ReLU (+ residual) backward in float64.  gs: list of [B, nvox, C] gradient contributions, y: raw
    conv output as stored, out: stored activation (its sign is the mask when a residual was added), else the mask is
    the sign of y a + b."""
    C = y.shape[2]
    cnt = float(y.shape[1] * C)
    mean, rstd = _mean_rstd32(stats, cnt)
    gam = gamma.double().view(1, 1, C)
    if out is not None:
        mask = out > 0
    else:
        a, b = _affine32(mean, rstd, gamma, beta)
        mask = (y * a + b) > 0
        del a, b
    dz = sum(gs) * mask
    dz_abs = sum(g.abs() for g in gs) * mask
    del mask
    xh = (y - mean) * rstd
    xh_abs = (y.abs() + mean.abs()) * rstd
    s1, s2 = (dz * gam).sum((1, 2)), (dz * gam * xh).sum((1, 2))
    a1 = (dz_abs * gam.abs()).sum((1, 2)) / cnt
    a2 = (dz_abs * gam.abs() * xh_abs).sum((1, 2)) / cnt
    r = {'dz': dz, 'dz_mag': dz_abs,
         'dgamma': (dz * xh).sum((0, 1)), 'dgamma_mag': (dz_abs * xh_abs).sum((0, 1)),
         'dbeta': dz.sum((0, 1)), 'dbeta_mag': dz_abs.sum((0, 1))}
    r['dy'] = rstd * (gam * dz - (s1 / cnt).view(-1, 1, 1) - xh * (s2 / cnt).view(-1, 1, 1))
    del xh
    r['dy_mag'] = rstd * (gam.abs() * dz_abs + a1.view(-1, 1, 1) + xh_abs * a2.view(-1, 1, 1))
    r['dbias'], r['dbias_mag'] = r['dy'].sum((0, 1)), r['dy_mag'].sum((0, 1))
    return r


def wgrad_reference(mode, x, gy):
    """weight gradient in the parameter layout (K3 / K2S2: [Co, Ci, k, k, k], T2S2: [Ci, Co, 2, 2, 2]) as one float64
    matmul per tap; x [B, D, H, W, Ci], gy [B, Do, Ho, Wo, Co]"""
    from segmentation3d._b200 import lib
    Ci, Co = x.shape[-1], gy.shape[-1]
    k = 3 if mode == lib.CONV_K3 else 2
    shape = (Ci, Co, k, k, k) if mode == lib.CONV_T2S2 else (Co, Ci, k, k, k)
    ref, mag = x.new_zeros(shape), x.new_zeros(shape)
    D, H, W = x.shape[1:4]
    if mode == lib.CONV_K3:
        xp = F.pad(x, (0, 0, 1, 1, 1, 1, 1, 1))
    g2 = gy.reshape(-1, Co)
    ga = g2.abs()
    for (a, b, c) in _taps(k):
        if mode == lib.CONV_T2S2:
            xs, gs = x.reshape(-1, Ci), gy[:, a::2, b::2, c::2].reshape(-1, Co)
            ref[:, :, a, b, c], mag[:, :, a, b, c] = xs.t() @ gs, xs.abs().t() @ gs.abs()
            continue
        if mode == lib.CONV_K3:
            xs = xp[:, a:a + D, b:b + H, c:c + W].reshape(-1, Ci)
        else:
            xs = x[:, a::2, b::2, c::2].reshape(-1, Ci)
        ref[:, :, a, b, c], mag[:, :, a, b, c] = (xs.t() @ g2).t(), (xs.abs().t() @ ga).t()
    return ref, mag


def dgrad_reference(mode, gy, w, xdims):
    """data gradient [B, D, H, W, Ci] of a convolution with parameter w (layout as above) from gy [B, Do, Ho, Wo, Co]"""
    from segmentation3d._b200 import lib
    B, Co = gy.shape[0], gy.shape[-1]
    D, H, W = xdims
    g2 = gy.reshape(-1, Co)
    if mode == lib.CONV_K3:
        Ci = w.shape[1]
        out = gy.new_zeros((B, D + 2, H + 2, W + 2, Ci))
        for (a, b, c) in _taps(3):
            out[:, a:a + D, b:b + H, c:c + W] += (g2 @ w[:, :, a, b, c]).view(B, D, H, W, Ci)
        return out[:, 1:D + 1, 1:H + 1, 1:W + 1]
    if mode == lib.CONV_K2S2:
        Ci = w.shape[1]
        out = gy.new_zeros((B, D, H, W, Ci))
        for (a, b, c) in _taps(2):
            out[:, a::2, b::2, c::2] = (g2 @ w[:, :, a, b, c]).view(B, D // 2, H // 2, W // 2, Ci)
        return out
    Ci = w.shape[0]
    out = gy.new_zeros((B, D, H, W, Ci))
    for (a, b, c) in _taps(2):
        out += (gy[:, a::2, b::2, c::2].reshape(-1, Co) @ w[:, :, a, b, c].t()).view(B, D, H, W, Ci)
    return out


def tail_reference(y, stats1, stats2, g1, b1, w2, bias2, g2, b2, dprobs):
    """out-block tail (GN1 -> ReLU -> 1x1x1 conv -> GN2 -> softmax) backward in float64.  y: [B, nvox, C] raw conv1
    output as stored, stats: [B, 2] forward sums, dprobs [B, C, nvox].  Returns outputs and magnitudes."""
    B, nv, C = y.shape
    cnt = float(nv * C)
    mean1, rstd1 = _mean_rstd32(stats1, cnt)
    mean2, rstd2 = _mean_rstd32(stats2, cnt)
    a1, c1 = _affine32(mean1, rstd1, g1, b1)
    a2, c2 = _affine32(mean2, rstd2, g2, b2)
    u = y * a1 + c1
    mask = u > 0
    h = u * mask
    h_abs = (y.abs() * a1.abs() + c1.abs()) * mask
    W2 = w2.double().reshape(C, C)
    z = h @ W2.t() + bias2.double().view(1, 1, C)
    z_abs = h_abs @ W2.abs().t() + bias2.double().abs().view(1, 1, C)
    xh2 = (z - mean2) * rstd2
    xh2_abs = (z_abs + mean2.abs()) * rstd2
    p = torch.softmax(z * a2 + c2, 2)
    dp = dprobs.double().reshape(B, C, nv).transpose(1, 2)
    dl = p * (dp - (p * dp).sum(2, keepdim=True))
    dl_abs = p * (dp.abs() + (p * dp.abs()).sum(2, keepdim=True))
    G2, G1 = g2.double().view(1, 1, C), g1.double().view(1, 1, C)

    def gn_back(dz, dz_abs, xh, xh_abs, rstd, G):
        s1, s2 = (G * dz).sum((1, 2)), (G * dz * xh).sum((1, 2))
        m1, m2 = (G.abs() * dz_abs).sum((1, 2)) / cnt, (G.abs() * dz_abs * xh_abs).sum((1, 2)) / cnt
        d = rstd * (G * dz - (s1 / cnt).view(-1, 1, 1) - xh * (s2 / cnt).view(-1, 1, 1))
        d_abs = rstd * (G.abs() * dz_abs + m1.view(-1, 1, 1) + xh_abs * m2.view(-1, 1, 1))
        return d, d_abs

    r = {'gn2.weight': ((dl * xh2).sum((0, 1)), (dl_abs * xh2_abs).sum((0, 1))),
         'gn2.bias': (dl.sum((0, 1)), dl_abs.sum((0, 1)))}
    dz2, dz2_abs = gn_back(dl, dl_abs, xh2, xh2_abs, rstd2, G2)
    r['conv2.bias'] = (dz2.sum((0, 1)), dz2_abs.sum((0, 1)))
    r['conv2.weight'] = (torch.einsum('bvo,bvc->oc', dz2, h), torch.einsum('bvo,bvc->oc', dz2_abs, h_abs))
    dg1, dg1_abs = (dz2 @ W2) * mask, (dz2_abs @ W2.abs()) * mask
    xh1 = (y - mean1) * rstd1
    xh1_abs = (y.abs() + mean1.abs()) * rstd1
    r['gn1.weight'] = ((dg1 * xh1).sum((0, 1)), (dg1_abs * xh1_abs).sum((0, 1)))
    r['gn1.bias'] = (dg1.sum((0, 1)), dg1_abs.sum((0, 1)))
    dy1, dy1_abs = gn_back(dg1, dg1_abs, xh1, xh1_abs, rstd1, G1)
    r['conv1.bias'] = (dy1.sum((0, 1)), dy1_abs.sum((0, 1)))
    r['dy1'] = (dy1, dy1_abs)
    r['z'] = (z, z_abs)
    return r


def check_stats(name, stats, y):
    """forward GroupNorm sums (accumulated from the unrounded conv output) against the stored, bf16-rounded tensor:
    each stored value is within 2^-8 of the summed one, its square within 2^-7 (+ 2^-16)"""
    y = y.flatten(1)
    st = stats.double()
    ref0, ref1 = y.sum(1), (y * y).sum(1)
    assert bool(((st[:, 0] - ref0).abs() <= BF16_REL * y.abs().sum(1)).all()), (name, 'sum', st[:, 0], ref0)
    assert bool(((st[:, 1] - ref1).abs() <= 2.01 * BF16_REL * ref1).all()), (name, 'sum of squares', st[:, 1], ref1)


# ---- the real run ---------------------------------------------------------------------------------------------------
_RUNS = {}


def run_case(case):
    """one bf16 training forward + backward through the autograd path train_step uses; the workspace of that step"""
    if case in _RUNS:
        return _RUNS[case]
    _RUNS.clear()                       # one case's buffers at a time
    arch, C, lossname, B, D, H, W = case
    from segmentation3d.loss.cross_entropy_loss import CrossEntropyLoss
    from segmentation3d.loss.focal_loss import FocalLoss
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, C, 0), 5)
    net = importlib.import_module('segmentation3d.network.' + arch).SegmentationNet(1, C)
    net.load_state_dict(sd)
    net.b200_mode = 'bf16'
    net = net.cuda().train()
    g = torch.Generator().manual_seed(B + D + 7 * C)
    crops = torch.randn((B, 1, D, H, W), generator=g).cuda()
    masks = torch.randint(0, C, (B, 1, D, H, W), generator=g).float().cuda()
    lf = {'dice': lambda: MultiDiceLoss([1.0 / C] * C, C, True), 'focal': lambda: FocalLoss(C, alpha=[1.0] * C, gamma=2, use_gpu=True),
          'ce': lambda: CrossEntropyLoss()}[lossname]()
    probs = net(crops)
    captured = []
    probs.register_hook(lambda gr: captured.append(gr.detach().clone()))
    lf(probs, masks).backward()
    torch.cuda.synchronize()
    plan = net._plan
    assert plan.mode == 'bf16'
    ws, _ = plan.plan(B, D, H, W, train=True)
    bw = ws['bwd']
    grads = {n: p.grad.detach() for n, p in net.named_parameters()}
    params = {n: p.detach() for n, p in net.named_parameters()}
    _RUNS[case] = r = {'net': net, 'plan': plan, 'ws': ws, 'bw': bw, 'grads': grads, 'params': params,
                       'dprobs': captured[0], 'case': case}
    return r


def _contains(view, out):
    if view is None or view.buf is not out.buf:
        return False
    if view.off <= out.off and out.off + out.C <= view.off + view.C:
        return True
    assert out.off + out.C <= view.off or view.off + view.C <= out.off, 'partial channel overlap'
    return False


def consumers(r, u):
    """[(consumer, gradient window)] of unit u's output, from the channel spans of the workspace views"""
    ws, bw = r['ws'], r['bw']
    o = u['out']
    found = []
    for v in ws['units']:
        if _contains(v['x'], o):
            assert v['conv'] in bw.gd, ('a consumer without a data-gradient buffer', v['conv'])
            found.append((v['conv'] + '.x', _window(bw.gd[v['conv']], o.off - v['x'].off, o.C)))
        if _contains(v['res'], o):
            found.append((v['conv'] + '.res', _window(bw.dres[v['conv']], o.off - v['res'].off, o.C)))
    if _contains(ws['tail']['x'], o):
        found.append(('tail.x', _window(bw.gd_tail, o.off - ws['tail']['x'].off, o.C)))
    return found


def has_producer(ws, u):
    return any(_contains(u['x'], v['out']) for v in ws['units'])


def _x5(r, u):
    """the conv input the weight gradient read, [B, D, H, W, Ci] float64"""
    from segmentation3d._b200 import lib
    ws = r['ws']
    B = ws['B']
    D, H, W = ws['dims'][u['lin']]
    if u.get('xpad') is not None:          # input block: row-padded single-channel input
        xp = ws['x_in'].view(B, D, H, W + lib.CIN1_PAD)
        return xp[..., lib.CIN1_LEFT:lib.CIN1_LEFT + W].double().unsqueeze(-1)
    return _rows(u['x'], D * H * W).view(B, D, H, W, u['x'].C)


def gn_stage(r, u, gsrc):
    plan, ws, bw = r['plan'], r['ws'], r['bw']
    nv = ws['vox'][u['lout']]
    gnp = plan.gns[u['gn']]
    stats = ws['stats'][plan.gn_index[u['gn']]]
    y = _rows(u['raw'], nv)
    out = _rows(u['out'], nv) if u['res'] is not None else None
    ref = gn_reference([_rows(gv, nv) for gv in gsrc], y, stats, gnp.gamma, gnp.beta, out)
    name = u['conv']
    check_bf16(name + ' gy', _rows(bw.gy[name], nv), ref['dy'], ref['dy_mag'])
    if u['res'] is not None:
        check_bf16(name + ' dres', _rows(bw.dres[name], nv), ref['dz'], ref['dz_mag'])
    g = r['grads']
    check_f32(u['gn'] + '.weight grad', g[u['gn'] + '.weight'], ref['dgamma'], ref['dgamma_mag'])
    check_f32(u['gn'] + '.bias grad', g[u['gn'] + '.bias'], ref['dbeta'], ref['dbeta_mag'])
    check_f32(name + '.bias grad', g[name + '.bias'], ref['dbias'], ref['dbias_mag'])


def wgrad_stage(r, u, gy=None, frac=None):
    ws = r['ws']
    plan = r['plan']
    c = plan.convs[u['conv']]
    B = ws['B']
    od = ws['dims'][u['lout']]
    if gy is None:
        gy = _rows(r['bw'].gy[u['conv']], ws['vox'][u['lout']])
    gy = gy.view(B, od[0], od[1], od[2], -1)[..., :c.real_cout]
    ref, mag = wgrad_reference(c.mode, _x5(r, u), gy)
    got = r['grads'][u['conv'] + '.weight']
    frac = wgrad_bound(r, u) if frac is None else frac
    ratio = float(((got.double() - ref).abs() / (mag + 1e-300)).max())
    r.setdefault('wgrad_log', []).append((u['conv'], ratio, frac))
    check_wgrad(u['conv'] + '.weight grad', got, ref, mag, frac)


def dgrad_stage(r, u, gy=None, gd=None):
    ws, bw, plan = r['ws'], r['bw'], r['plan']
    name = u['conv']
    c = plan.convs[name]
    B = ws['B']
    od, xd = ws['dims'][u['lout']], ws['dims'][u['lin']]
    if gy is None:
        gy = _rows(bw.gy[name], ws['vox'][u['lout']])
    gy = gy.view(B, od[0], od[1], od[2], -1)[..., :c.real_cout]
    # the data-gradient convolution reads the parameter rounded to its packed weight type
    w = r['params'][name + '.weight'].to(bw.dconv[name].w.dtype).double()
    ref = dgrad_reference(c.mode, gy, w, xd)
    mag = dgrad_reference(c.mode, gy.abs(), w.abs(), xd)
    if gd is None:
        gd = bw.gd[name]
    got = _rows(gd, ws['vox'][u['lin']]).view(ref.shape)
    check_bf16(name + ' gd', got, ref, mag)


def tail_stage(r):
    plan, ws, bw = r['plan'], r['ws'], r['bw']
    tail = ws['tail']
    nc, ncp, nv = plan.out_channels, tail['ncp'], ws['vox'][0]
    assert bw.gy_tail.ld == ncp and tail['raw'].ld == ncp
    g1, g2 = plan.gns['out_block.gn1'], plan.gns['out_block.gn2']
    y = _rows(_window(tail['raw'], 0, nc), nv)
    ref = tail_reference(y, ws['stats'][plan.gn_index['out_block.gn1']], ws['stats2'], g1.gamma, g1.beta, plan.w2, plan.b2,
                         g2.gamma, g2.beta, r['dprobs'])
    gy = _rows(bw.gy_tail, nv)
    check_bf16('out_block gy_tail', gy[..., :nc], *ref['dy1'])
    assert bool((gy[..., nc:] == 0).all()), 'padding channels of gy_tail must stay exactly 0'
    for k in ('gn2.weight', 'gn2.bias', 'conv2.bias', 'conv2.weight', 'gn1.weight', 'gn1.bias', 'conv1.bias'):
        got = r['grads']['out_block.' + k]
        check_f32('out_block.' + k + ' grad', got.reshape(ref[k][0].shape), *ref[k])
    return gy, ref


def tail_stats_stage(r, ref):
    plan, ws = r['plan'], r['ws']
    nc, nv = plan.out_channels, ws['vox'][0]
    check_stats('out_block.gn1', ws['stats'][plan.gn_index['out_block.gn1']], _rows(_window(ws['tail']['raw'], 0, nc), nv))
    # the second GroupNorm's sums are formed in fp32 from the stored conv1 output (seg3d_outblock_tail_stats)
    z, z_abs = ref['z']
    st = ws['stats2'].double()
    assert bool(((st[:, 0] - z.sum((1, 2))).abs() <= BF16_MAG * z_abs.sum((1, 2))).all()), ('stats2 sum', st[:, 0], z.sum((1, 2)))
    assert bool(((st[:, 1] - (z * z).sum((1, 2))).abs() <= 2 * BF16_MAG * (z_abs * z_abs).sum((1, 2))).all()), 'stats2 sum of squares'


def expected_stages(ws):
    """per unit: forward sums, GroupNorm backward, weight gradient (+ data gradient when its input has a producer);
    the tail: its sums, its backward, conv1's weight and data gradients"""
    return 4 + sum(3 + int(has_producer(ws, u)) for u in ws['units'])


def _tail_unit(ws):
    return {'conv': 'out_block.conv1', 'x': ws['tail']['x'], 'lin': 0, 'lout': 0}


def check_all_stages(r):
    ws, plan = r['ws'], r['plan']
    n = 0
    arch = r['case'][0]
    gy_tail, tref = tail_stage(r)
    tail_stats_stage(r, tref)
    del tref
    wgrad_stage(r, _tail_unit(ws), gy_tail)
    dgrad_stage(r, _tail_unit(ws), gy_tail, r['bw'].gd_tail)
    n += 4
    del gy_tail
    counts = {}
    for u in ws['units']:
        nv = ws['vox'][u['lout']]
        check_stats(u['gn'], ws['stats'][plan.gn_index[u['gn']]], _rows(u['raw'], nv))
        cons = consumers(r, u)
        counts[u['conv']] = len(cons)
        assert 1 <= len(cons) <= 3, (u['conv'], [k for k, _ in cons])
        gn_stage(r, u, [gv for _, gv in cons])
        wgrad_stage(r, u)
        n += 3
        assert has_producer(ws, u) == (u['conv'] in r['bw'].gd), u['conv']
        if has_producer(ws, u):
            dgrad_stage(r, u)
            n += 1
    if arch == 'vnet':
        assert counts == VNET_CONSUMERS, counts
    return n


@pytest.mark.parametrize('case', CASES, ids=lambda c: '%s%d-%s-%dx%dx%dx%d' % c)
def test_every_backward_stage_matches_float64(case):
    r = run_case(case)
    r['wgrad_log'] = []
    n = check_all_stages(r)
    want = expected_stages(r['ws'])
    print('%s: %d backward stages checked against float64 (%d units)' % (str(case), n, len(r['ws']['units'])))
    print('  weight gradients, worst |err| / sum|x||dy| against the bound:')
    for name, ratio, frac in r['wgrad_log']:
        print('    %-28s %.2e  (bound %.2e)' % (name, ratio, frac))
    assert n == want, (n, want)


# weight gradients of the 8 x 96^3 step measured on B200 to miss the fp32 bound of the small shapes, 2e-5 sum |x| |dy|:
# up_32's conv (nine taps per MMA, ~1 100 tiles per CTA) by 4x, up_64's first block conv (~430 tiles per CTA) by 13x
FP32_BOUND_MISSES = ['up_32.rblock.ops.0.conv', 'up_64.rblock.ops.0.conv']


# an expected failure of the kernels: the CPU dry run (tests/dryrun_gpu_tests_on_cpu.py) emulates them exactly and meets it
@pytest.mark.xfail(torch.cuda.is_available(), strict=True, reason='one wave of CTAs, each summing hundreds of tiles in one truncating fp32 tensor-memory '
                                       'accumulator (DESIGN section 2); turns red once the kernels meet the bound')
@pytest.mark.parametrize('name', FP32_BOUND_MISSES)
def test_bench_step_weight_gradients_meet_the_fp32_bound(name):
    """Open finding: at the benchmarked step these weight gradients stay inside the bound derived from their kernels'
    accumulation length (wgrad_bound, checked above) but not inside the 2e-5 an fp32 sum meets at the small shapes, and
    their error exceeds the effect of one dropped 512-voxel chunk at level 0.  Capping the tiles per CTA fixes it but cost
    2-6 % of the training step on B200; draining the accumulator every few hundred steps would keep the rate."""
    r = run_case(BENCH)
    wgrad_stage(r, _unit(r, name), frac=F32_MAG)


# ---- the checks can fail --------------------------------------------------------------------------------------------
def _unit(r, name):
    return next(u for u in r['ws']['units'] if u['conv'] == name)


@pytest.mark.parametrize('defect', ['gd_plane_zeroed', 'wgrad_chunk_dropped', 'concat_halves_swapped'])
def test_stage_checks_reject_injected_defects(defect):
    """Perturbed copies of real buffers of the 8 x 96^3 step go through the same comparisons and must be rejected:
    one z-plane of a data gradient zeroed at a z-tile seam; the contribution of one fixed 512-voxel chunk (sample 0, the
    first one of z-plane 16) taken out of the kernel's weight gradient of up_128's first block conv, at level 2 where the
    derived bound (~1.4e-4) resolves a chunk - at level 0 it does not (~1e-3 against ~7e-5 per chunk), which is the finding
    of the test above; the halves of a concat producer's gradient windows swapped."""
    from segmentation3d._b200.plan import _View
    r = run_case(BENCH)
    ws, bw = r['ws'], r['bw']
    if defect == 'gd_plane_zeroed':
        u = _unit(r, 'up_32.rblock.ops.0.conv')
        g = bw.gd[u['conv']]
        bad = g.buf.clone()
        D, H, W = ws['dims'][0]
        bad.view(ws['B'], D, H, W, -1)[:, D // 2] = 0
        dgrad_stage(r, u)                                     # the real buffer passes
        with pytest.raises(AssertionError, match=r'up_32\.rblock\.ops\.0\.conv gd: \d+ of'):
            dgrad_stage(r, u, gd=_View(bad, g.off, g.ld, g.C))
    elif defect == 'wgrad_chunk_dropped':
        u = _unit(r, 'up_128.rblock.ops.0.conv')
        B = ws['B']
        D, H, W = ws['dims'][u['lin']]
        x = _x5(r, u)
        gy = _rows(bw.gy[u['conv']], D * H * W).view(B, D, H, W, -1)
        ref, mag = wgrad_reference(r['plan'].convs[u['conv']].mode, x, gy)
        frac = wgrad_bound(r, u)
        got = r['grads'][u['conv'] + '.weight'].double()
        check_wgrad(u['conv'] + '.weight grad', got, ref, mag, frac)        # the kernel's gradient passes
        lo = 16 * H * W
        assert lo % 512 == 0
        xp = F.pad(x[:1], (0, 0, 1, 1, 1, 1, 1, 1))
        g0 = gy[0].reshape(-1, gy.shape[-1])[lo:lo + 512]
        bad = got.clone()
        for (a, b, c) in _taps(3):
            xs = xp[0, a:a + D, b:b + H, c:c + W].reshape(-1, x.shape[-1])[lo:lo + 512]
            bad[:, :, a, b, c] -= (xs.t() @ g0).t()
        with pytest.raises(AssertionError, match=r'up_128\.rblock\.ops\.0\.conv\.weight grad: \d+ of'):
            check_wgrad(u['conv'] + '.weight grad', bad, ref, mag, frac)
    else:
        u = _unit(r, 'up_32.up_conv')                         # the lower half of the level-0 concat buffer
        cons = consumers(r, u)
        assert len(cons) == 2 and u['out'].off == 0
        gn_stage(r, u, [gv for _, gv in cons])
        swapped = [_window(gv, u['out'].C, u['out'].C) for _, gv in cons]      # the skip half's windows instead
        with pytest.raises(AssertionError, match=r'up_32\.up_conv gy: \d+ of'):
            gn_stage(r, u, swapped)


# ---- seg3d_outblock_tail_bwd on synthetic data ----------------------------------------------------------------------
TAIL_CASES = [(C, ld, nvox, dt) for C in (1, 2, 3, 7, 16) for ld in sorted({C, 16}) for nvox in (1024, 1000)
              for dt in ('BF16', 'F32')]


@pytest.mark.parametrize('C,ld,nvox,dt_name', TAIL_CASES, ids=lambda v: str(v))
def test_outblock_tail_bwd_matches_float64(C, ld, nvox, dt_name):
    """all three passes of seg3d_outblock_tail_bwd against the float64 tail backward, with the kernel's ReLU mask and the
    bounds above; the padding channels of the gradient buffer are not written"""
    from segmentation3d._b200 import lib as L
    L.load()
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    B = 3
    g = torch.Generator().manual_seed(100 * C + ld + nvox)
    yb = (torch.randn((B, nvox, ld), generator=g) * 2.0 + 0.5).to(tdt).cuda()
    y = yb[..., :C].double()
    stats1 = torch.stack([y.flatten(1).sum(1), (y * y).flatten(1).sum(1)], 1).contiguous()
    gamma1, beta1 = (torch.rand(C, generator=g) + 0.5).cuda(), (torch.randn(C, generator=g) * 0.3).cuda()
    w2, bias2 = (torch.randn((C, C), generator=g) / C ** 0.5).cuda(), (torch.randn(C, generator=g) * 0.1).cuda()
    gamma2, beta2 = (torch.rand(C, generator=g) + 0.5).cuda(), (torch.randn(C, generator=g) * 0.3).cuda()
    dprobs = (torch.randn((B, C, nvox), generator=g) * 1e-3).cuda()
    # the second GroupNorm's forward sums: any consistent input; the float64 conv2 output of the reference
    zero = torch.zeros((B, 2), dtype=torch.float64).cuda()
    z = tail_reference(y, stats1, zero + 1.0, gamma1, beta1, w2, bias2, gamma2, beta2, dprobs)['z'][0]
    stats2 = torch.stack([z.flatten(1).sum(1), (z * z).flatten(1).sum(1)], 1).contiguous()
    ref = tail_reference(y, stats1, stats2, gamma1, beta1, w2, bias2, gamma2, beta2, dprobs)
    sums2, sums1 = zero.clone(), zero.clone()
    outs = {k: torch.zeros((n,), dtype=torch.float32).cuda() for k, n in
            (('gn2.weight', C), ('gn2.bias', C), ('conv2.weight', C * C), ('conv2.bias', C), ('gn1.weight', C), ('gn1.bias', C),
             ('conv1.bias', C))}
    dy = torch.zeros((B, nvox, ld), dtype=tdt).cuda()
    for p in range(3):
        L.call('seg3d_outblock_tail_bwd', dt, p, L.ptr(yb), ld, C, L.ptr(stats1), L.ptr(gamma1), L.ptr(beta1), L.ptr(w2),
               L.ptr(bias2), L.ptr(stats2), L.ptr(gamma2), L.ptr(beta2), 1e-5, L.ptr(dprobs), L.ptr(sums2), L.ptr(sums1),
               L.ptr(outs['gn2.weight']), L.ptr(outs['gn2.bias']), L.ptr(outs['conv2.weight']), L.ptr(outs['conv2.bias']),
               L.ptr(outs['gn1.weight']), L.ptr(outs['gn1.bias']), L.ptr(outs['conv1.bias']), L.ptr(dy), ld, B, nvox,
               L.stream_ptr())
    torch.cuda.synchronize()
    if dt_name == 'BF16':
        check_bf16('dy1', dy[..., :C], *ref['dy1'])
    else:
        _close('dy1', dy[..., :C], ref['dy1'][0], ref['dy1'][1], 0.0, BF16_MAG)
    assert bool((dy[..., C:] == 0).all()), 'padding channels written'
    for k, got in outs.items():
        check_f32(k, got.reshape(ref[k][0].shape), *ref[k])
