"""Nets with more than 16 classes on the GPU: the tensor-core out-block tail (csrc/tail_wide.cu, seg3d_outblock_tail_wide)
against float64, against the SIMT tail where both apply, and the whole inference stack (plan, sliding window, seg_infer,
the standalone OutputBlock) against the oracle.

Error bound of the kernel, derived from its accumulation: h = relu(fma(raw, a1, b1)) is formed in fp32 as the SIMT tail
forms it (|dh| <= 2^-22 (|raw a1| + |beta1| + |mean1 a1|), the fold's and the fma's roundings); h = hi + lo and
w2 = whi + wlo in f16 drop lo * wlo and round lo / wlo (<= 3 * 2^-22 |w||h| per product, plus 2^-25 absolute for an f16
subnormal); the 3 * Cp / 16 MMAs of K = 16 add into the fp32 accumulator with truncation, one more rounding for the bias:
    |dz| <= ((3 Cp / 16 + 2) 2^-23 + 3 * 2^-22) sum|w2||h| + 2^-24 (sum|h| + |b2|) + sum|w2||dh|.
The GN2 sums add each epilogue thread's z (and z^2) in fp32 before the fp64 atomics: k terms per thread add k 2^-24 of
the summed magnitudes.  The logits l = fma(z, a2, b2) carry |a2||dz| plus the fold's roundings; a softmax output moves by
at most p (2 max|dl| + 2^-23 (|l| + max|l|) + (C + 8) 2^-23) (exp, sum, reciprocal and product roundings)."""
import importlib
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from oracle import net as onet
from oracle import sliding_window as osw

pytestmark = pytest.mark.gpu
EPS = 1e-5
U = 2.0 ** -24


@pytest.fixture(scope='module')
def lib():
    from segmentation3d._b200 import lib as L
    L.load()
    return L


def _fold(st, nvox, C, gamma, beta):
    """GroupNorm(1, C) folded per sample as gn_mean_rstd + the kernels do: a = fp32(rstd * gamma), b = beta - mean * a;
    returns float64 a, b [N, C] and the magnitude |beta| + |mean a| that the fold's rounding scales with"""
    cnt = float(nvox * C)
    m = st[:, 0].double() / cnt
    var = (st[:, 1].double() / cnt - m * m).clamp_min(0)
    mean = m.float()
    rstd = (1.0 / torch.sqrt(var + EPS)).float()
    a = (rstd[:, None] * gamma.float()[None, :]).double()
    ma = mean.double()[:, None] * a
    return a, beta.double()[None, :] - ma, beta.double().abs()[None, :] + ma.abs()


def _z_ref(x, nid, fold1, w2, b2, Cp):
    """float64 z = conv2(relu(gn1(raw))) of raw rows x [M, C] (samples nid [M]) and the kernel's bound on |dz|"""
    a1, b1, f1 = fold1
    xd = x.double()
    xa = xd * a1[nid]
    h = (xa + b1[nid]).clamp_min(0)
    eh = 4 * U * (xa.abs() + f1[nid])
    W = w2.double()
    Wa = W.abs()
    z = h @ W.t() + b2.double()[None, :]
    ez = (((3 * Cp / 16 + 2) * 2 * U + 3 * 4 * U) * (h @ Wa.t()) + U * (h.sum(1, keepdim=True) + b2.double().abs()[None, :])
          + eh @ Wa.t())
    return z, ez


def _p_ref(z, ez, nid, fold2, C):
    a2, b2, f2 = fold2
    za = z * a2[nid]
    l = za + b2[nid]
    el = a2[nid].abs() * ez + 4 * U * (za.abs() + f2[nid])
    p = torch.softmax(l, 1)
    m = l.abs().max(1, keepdim=True).values
    ep = p * (2 * el.max(1, keepdim=True).values + 2 * U * (l.abs() + m) + (C + 8) * 2 * U) + 1e-30
    return p, ep


def _params(C, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)

    def r(*s):
        return torch.randn(s, generator=g, device='cuda')
    return {'g1': 1 + 0.3 * r(C), 'b1': 0.2 * r(C), 'w2': r(C, C) * (2.0 / C) ** 0.5, 'bias2': 0.2 * r(C),
            'g2': 1 + 0.3 * r(C), 'b2': 0.2 * r(C)}


def _raw(N, nvox, C, ld, seed):
    """fp32 rows [N][nvox][ld]; channels >= C are NaN so a read of them shows"""
    g = torch.Generator(device='cuda').manual_seed(seed)
    raw = torch.full((N, nvox, ld), float('nan'), device='cuda')
    raw[..., :C] = torch.randn((N, nvox, C), generator=g, device='cuda') * 0.8 + 0.3
    x = raw[..., :C].double()
    st1 = torch.stack([x.sum((1, 2)), (x * x).sum((1, 2))], 1).contiguous()
    return raw, st1


def _acc_terms(C, N, nvox):
    """fp32 terms one epilogue thread of the wide kernel adds before its warp sum (contiguous tiles per CTA, 3 groups)"""
    ntiles = N * ((nvox + 127) // 128)
    grid = min(ntiles, torch.cuda.get_device_properties(0).multi_processor_count)
    per_cta = (ntiles + grid - 1) // grid
    return C * ((per_cta + 2) // 3) + 40


def _run_wide(lib, ps, raw, ld, C, st1, P, st2, probs, N, nvox):
    lib.call('seg3d_outblock_tail_wide', ps, lib.ptr(raw), ld, C, lib.ptr(st1), lib.ptr(P['g1']), lib.ptr(P['b1']),
             lib.ptr(P['w2']), lib.ptr(P['bias2']), EPS, lib.ptr(st2), lib.ptr(P['g2']), lib.ptr(P['b2']),
             lib.ptr(probs), N, nvox, lib.stream_ptr())


def _check_stats(st2, raw, st1, P, C, Cp, N, nvox, kacc, extra=None):
    fold1 = _fold(st1, nvox, C, P['g1'], P['b1'])
    for n in range(N):
        x = raw[n, :, :C]
        nid = torch.full((nvox,), n, dtype=torch.long, device='cuda')
        z, ez = _z_ref(x, nid, fold1, P['w2'], P['bias2'], Cp)
        if extra is not None:
            ez = ez + extra(x, nid, fold1)
        s, ss = float(z.sum()), float((z * z).sum())
        es = float(ez.sum()) + kacc * U * float(z.abs().sum())
        ess = float((2 * z.abs() * ez + ez * ez).sum()) + kacc * U * float((z * z).sum())
        assert abs(float(st2[n, 0]) - s) <= es, (C, n, float(st2[n, 0]), s, es)
        assert abs(float(st2[n, 1]) - ss) <= ess, (C, n, float(st2[n, 1]), ss, ess)


def _check_probs(probs, raw, st1, st2, P, C, Cp, N, nvox, vox_idx=None):
    fold1 = _fold(st1, nvox, C, P['g1'], P['b1'])
    fold2 = _fold(st2, nvox, C, P['g2'], P['b2'])
    worst = 0.0
    for n in range(N):
        v = torch.arange(nvox, device='cuda') if vox_idx is None else vox_idx
        nid = torch.full((v.numel(),), n, dtype=torch.long, device='cuda')
        z, ez = _z_ref(raw[n, v, :C], nid, fold1, P['w2'], P['bias2'], Cp)
        p, ep = _p_ref(z, ez, nid, fold2, C)
        got = probs[n][:, v].t().double()
        d = (got - p).abs()
        assert bool((d <= ep).all()), (C, n, float(d.max()), float((d - ep).max()))
        assert float((got.sum(1) - 1).abs().max()) <= 1e-5
        worst = max(worst, float(d.max()))
    return worst


KERNEL_CASES = [(C, N, nvox, pad) for C in (17, 31, 32, 48, 64, 100, 127) for N in (1, 3) for nvox in (1000, 4096, 24576)
                for pad in (0, 8)]


@pytest.mark.parametrize('C,N,nvox,pad', KERNEL_CASES)
def test_wide_tail_kernel_against_float64(lib, C, N, nvox, pad):
    Cp = (C + 15) // 16 * 16
    ld = Cp + pad
    seed = C * 1000 + N * 100 + nvox % 97 + pad
    raw, st1 = _raw(N, nvox, C, ld, seed)
    P = _params(C, seed + 1)
    st2 = torch.full((N + 1, 2), 12345.0, dtype=torch.float64, device='cuda')
    st2[:N] = 0
    total = N * C * nvox
    probs = torch.full((total + 4096,), float('nan'), device='cuda')
    nan_bits = probs[-1:].view(torch.int32).clone()
    _run_wide(lib, 0, raw, ld, C, st1, P, st2, probs, N, nvox)
    torch.cuda.synchronize()
    assert bool(probs.isnan().all()), 'pass 0 writes no probabilities'
    _check_stats(st2, raw, st1, P, C, Cp, N, nvox, _acc_terms(C, N, nvox))
    st2_after0 = st2.clone()
    _run_wide(lib, 1, raw, ld, C, st1, P, st2, probs, N, nvox)
    torch.cuda.synchronize()
    assert torch.equal(st2, st2_after0) and float(st2[N, 0]) == 12345.0          # pass 1 reads the sums, writes nothing else
    assert not bool(probs[:total].isnan().any()), 'every probability is written'
    assert bool((probs[total:].view(torch.int32) == nan_bits).all()), 'nothing past [N, C, nvox] changes'
    worst = _check_probs(probs[:total].view(N, C, nvox), raw, st1, st2[:N], P, C, Cp, N, nvox)
    print('C=%d N=%d nvox=%d ld=%d max|dp| %.3g' % (C, N, nvox, ld, worst))


@pytest.mark.parametrize('C', list(range(2, 17)))
def test_wide_tail_computes_the_simt_tail(lib, C):
    """C = 2..16, where the SIMT tail (seg3d_outblock_tail_stats / _probs, exact fp32 FMA chains) also runs: the two agree
    within the sum of their bounds (the SIMT z: C + 2 roundings of sum|w2||h|; its sums: one value per thread per voxel,
    reduced in fp32 over a 256-thread block)"""
    N, nvox = 3, 24576 + 77
    Cp = (C + 15) // 16 * 16
    ld = Cp
    raw, st1 = _raw(N, nvox, C, ld, 7 + C)
    raw[..., C:] = 0              # the SIMT tail takes ld >= C and reads channels < C only, as the wide one does
    P = _params(C, 11 + C)
    total = N * C * nvox
    st2w = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    st2s = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    pw = torch.empty(total, device='cuda')
    ps = torch.empty(total, device='cuda')
    _run_wide(lib, 0, raw, ld, C, st1, P, st2w, pw, N, nvox)
    lib.call('seg3d_outblock_tail_stats', lib.F32, lib.ptr(raw), ld, C, lib.ptr(st1), lib.ptr(P['g1']), lib.ptr(P['b1']),
             lib.ptr(P['w2']), lib.ptr(P['bias2']), EPS, lib.ptr(st2s), N, nvox, lib.stream_ptr())
    _run_wide(lib, 1, raw, ld, C, st1, P, st2w, pw, N, nvox)
    lib.call('seg3d_outblock_tail_probs', lib.F32, lib.ptr(raw), ld, C, lib.ptr(st1), lib.ptr(P['g1']), lib.ptr(P['b1']),
             lib.ptr(P['w2']), lib.ptr(P['bias2']), lib.ptr(st2w), lib.ptr(P['g2']), lib.ptr(P['b2']), EPS, lib.ptr(ps), N, nvox,
             lib.stream_ptr())
    torch.cuda.synchronize()
    fold1 = _fold(st1, nvox, C, P['g1'], P['b1'])
    fold2 = _fold(st2w, nvox, C, P['g2'], P['b2'])
    kw = _acc_terms(C, N, nvox)
    for n in range(N):
        nid = torch.full((nvox,), n, dtype=torch.long, device='cuda')
        z, ez = _z_ref(raw[n, :, :C], nid, fold1, P['w2'], P['bias2'], Cp)
        xa = raw[n, :, :C].double() * fold1[0][nid]
        h = (xa + fold1[1][nid]).clamp_min(0)
        ezs = (C + 2) * U * (h @ P['w2'].double().abs().t() + P['bias2'].double().abs()[None, :]) + \
            4 * U * (xa.abs() + fold1[2][nid]) @ P['w2'].double().abs().t()
        za = z.abs()
        es = float((ez + ezs).sum()) + (kw + C + 300) * U * float(za.sum())
        ess = float((2 * za * (ez + ezs) + (ez + ezs) ** 2).sum()) + (kw + C + 300) * U * float((z * z).sum())
        assert abs(float(st2w[n, 0] - st2s[n, 0])) <= es, (C, n, float(st2w[n, 0]), float(st2s[n, 0]), es)
        assert abs(float(st2w[n, 1] - st2s[n, 1])) <= ess, (C, n)
        pr, epw = _p_ref(z, ez, nid, fold2, C)
        _, eps_ = _p_ref(z, ezs, nid, fold2, C)
        gw = pw.view(N, C, nvox)[n].t().double()
        gs = ps.view(N, C, nvox)[n].t().double()
        assert bool(((gw - gs).abs() <= epw + eps_).all()), (C, n, float((gw - gs).abs().max()))
        assert bool(((gw - pr).abs() <= epw).all()), (C, n, float((gw - pr).abs().max()))


def _net_forward(arch, cout, sd, x, mode=None):
    mod = importlib.import_module('segmentation3d.network.' + arch)
    net = mod.SegmentationNet(1, cout)
    net.load_state_dict(sd)
    if mode is not None:
        net.b200_mode = mode
    net = net.cuda().eval()
    with torch.no_grad():
        y = net(x.cuda())
    torch.cuda.synchronize()
    return y.cpu(), net.resolve_mode()


def _smooth(seed, shape):
    g = torch.Generator().manual_seed(seed)
    lo = torch.randn((shape[0], shape[1]) + tuple(max(2, s // 8) for s in shape[2:]), generator=g)
    x = F.interpolate(lo, size=shape[2:], mode='trilinear', align_corners=False) * 2
    return x + 0.3 * torch.randn(shape, generator=g)


@pytest.mark.parametrize('arch', ['vnet', 'vbnet'])
@pytest.mark.parametrize('cout', [17, 32, 64, 127])
@pytest.mark.parametrize('mode,tol', [('fp32', 1e-3), ('fp32x', 1e-3), ('fp16', 1e-2)])
def test_wide_net_matches_the_oracle(lib, arch, cout, mode, tol):
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 3), 11)
    x = _smooth(17, (2, 1, 32, 32, 32))
    ref = onet.forward(sd, x)
    y, resolved = _net_forward(arch, cout, sd, x, mode)
    assert resolved == mode and tuple(y.shape) == (2, cout, 32, 32, 32)
    assert float((y.sum(1) - 1).abs().max()) <= 1e-5
    err = float((y - ref).abs().max())
    print(arch, cout, 'classes', mode, 'max|dp| %.3g' % err)
    assert err <= tol, (arch, cout, mode, err)
    if mode == 'fp32x':
        assert _net_forward(arch, cout, sd, x[:1])[1] == 'fp32x'          # the default mode of a multi-class net


def test_benchmark_shape_127_classes_tail_against_float64(lib):
    """VNet, 127 classes, fp16, the benchmark's 36 patches of 96^3: both tail launches of the forward checked in float64
    (the GN2 sums of every sample in full, the probabilities on a seeded sample of 10^6 voxels)"""
    from segmentation3d._b200.plan import NetPlan
    C, B, S = 127, 36, 96
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, C, 0), 5)
    p = NetPlan(sd, mode='fp16', device='cuda')
    g = torch.Generator(device='cuda').manual_seed(2)
    x = torch.randn((B, 1, S, S, S), generator=g, device='cuda')
    probs = p.forward(x)
    torch.cuda.synchronize()
    ws, _ = p.plan(B, S, S, S)
    assert [m['kind'] for m in ws['meta'] if m['name'].startswith('out_block.tail')] == ['tail_wide', 'tail_wide']
    rv = ws['tail']['raw']
    nvox = S ** 3
    raw = rv.buf.view(B, nvox, rv.ld)
    st1 = ws['stats'][p.gn_index['out_block.gn1']]
    st2 = ws['stats2']
    g1, g2 = p.gns['out_block.gn1'], p.gns['out_block.gn2']
    P = {'g1': g1.gamma, 'b1': g1.beta, 'w2': p.w2, 'bias2': p.b2, 'g2': g2.gamma, 'b2': g2.beta}
    _check_stats(st2, raw, st1, P, C, 128, B, nvox, _acc_terms(C, B, nvox))
    gs = torch.Generator(device='cuda').manual_seed(1234)
    per = 10 ** 6 // B + 1
    v = torch.randint(0, nvox, (per,), generator=gs, device='cuda')
    worst = _check_probs(probs.view(B, C, nvox), raw, st1, st2, P, C, 128, B, nvox, vox_idx=v)
    print('127 classes, 36 x 96^3, fp16: sampled max|dp| vs float64 %.3g' % worst)


def _model(arch, cout, sd, mode, norm, batch=3):
    from segmentation3d.core.seg_infer import make_model
    mod = importlib.import_module('segmentation3d.network.' + arch)
    net = mod.SegmentationNet(1, cout)
    net.load_state_dict(sd)
    net.b200_mode = mode
    return make_model(net.cuda().eval(), [1.0, 1.0, 1.0], norm, batch=batch)


def _labels_sd(cout, seed):
    """random-init net with randomised affines and a spread of conv2 biases, so many labels win somewhere"""
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, cout, seed), seed + 1)
    g = torch.Generator().manual_seed(seed + 2)
    sd['out_block.gn2.bias'] = 0.5 * torch.randn(sd['out_block.gn2.bias'].shape, generator=g)
    return sd


def test_sliding_window_twenty_classes_matches_the_oracle(lib):
    from segmentation3d.core.seg_infer import segmentation_volume
    from segmentation3d.utils.image3d import Image3d
    cout = 20
    sd = _labels_sd(cout, 21)
    vol = (_smooth(4, (1, 1, 48, 48, 64))[0, 0].numpy() * 100).astype(np.float32)
    nd = {'type': 0, 'mean': 0.0, 'stddev': 100.0, 'clip': False}
    model = _model('vnet', cout, sd, 'fp32x', nd)
    cfg = {'partition_type': 'SIZE', 'partition_size': [32, 32, 32], 'partition_stride': [16, 16, 16],
           'pick_largest_cc': False, 'remove_small_cc': 0}
    probs_im, mask_im = segmentation_volume(model, cfg, Image3d(vol), None, None, True)
    probs = np.stack([q.to_numpy() for q in probs_im], 0)
    mask = mask_im.to_numpy()
    ref_p, ref_m, _, _ = osw.segmentation_volume(sd, vol, [1.0, 1.0, 1.0], nd, 'SIZE', [32, 32, 32], [16, 16, 16], 16,
                                                 double_forward=False, faithful_copies=False)
    assert int(ref_m.max()) > 16, 'the oracle mask holds labels above 16'
    err = float(np.abs(probs - ref_p).max())
    agree = float((mask == ref_m).mean())
    print('sliding window, 20 classes, fp32x: max|dp| %.3g, agreement %.5f, labels %s' % (err, agree, np.unique(ref_m)))
    assert err <= 1e-3 and agree >= 0.999
    assert np.array_equal(mask, osw.argmax_first(probs))


def test_seg_infer_twenty_class_model_folder(lib, tmp_path):
    from oracle import postprocess as opp
    from segmentation3d.core.seg_infer import segmentation
    from segmentation3d.utils.image3d import Image3d, read_image, write_image
    import segmentation3d.config.infer_config as icfg_mod
    cout = 20
    sd = _labels_sd(cout, 31)
    chk = tmp_path / 'model' / 'fine' / 'checkpoints' / 'chk_1'
    os.makedirs(str(chk))
    nd = {'type': 0, 'mean': 0.0, 'stddev': 100.0, 'clip': False}
    torch.save({'epoch': 1, 'batch': 0, 'net': 'vnet', 'max_stride': 16, 'state_dict': sd, 'spacing': [1.0, 1.0, 1.0],
                'interpolation': 'LINEAR', 'in_channels': 1, 'out_channels': cout, 'crop_normalizers': [nd]},
               str(chk / 'params.pth'))
    text = open(icfg_mod.__file__).read()
    text += ("\n__C.general.single_scale = 'fine'\n__C.fine.partition_size = [32, 32, 32]\n"
             "__C.fine.partition_stride = [16, 16, 16]\n__C.fine.pick_largest_cc = True\n")
    open(str(tmp_path / 'model' / 'infer_config.py'), 'w').write(text)
    vol = (_smooth(6, (1, 1, 48, 48, 64))[0, 0].numpy() * 100).astype(np.float32)
    os.makedirs(str(tmp_path / 'data'))
    write_image(Image3d(vol), str(tmp_path / 'data' / 'im.mha'), True)
    out = tmp_path / 'out'
    masks = segmentation(str(tmp_path / 'data' / 'im.mha'), str(tmp_path / 'model'), str(out), 'seg.mha', 0, True, True,
                         False, True)
    case = out / 'im.mha'
    assert sorted(os.listdir(str(case))) == sorted(['mean_prob_%d.mha' % c for c in range(cout)] + ['seg.mha'])
    seg = read_image(str(case / 'seg.mha')).to_numpy()
    probs = np.stack([read_image(str(case / ('mean_prob_%d.mha' % c))).to_numpy() for c in range(cout)], 0)
    assert seg.dtype == np.int8 and np.array_equal(seg, masks[0].to_numpy())
    assert float(np.abs(probs.sum(0) - 1).max()) <= 1e-5
    raw_mask = osw.argmax_first(probs)
    assert int(raw_mask.max()) > 16, 'labels above 16 are present before the filtering'
    assert np.array_equal(seg, opp.pick_largest_connected_component(raw_mask, list(range(1, cout))))
    ref_p, ref_m, _, _ = osw.segmentation_volume(sd, vol, [1.0, 1.0, 1.0], nd, 'SIZE', [32, 32, 32], [16, 16, 16], 16,
                                                 double_forward=False, faithful_copies=False)
    assert float(np.abs(probs - ref_p).max()) <= 1e-3 and float((raw_mask == ref_m).mean()) >= 0.999


@pytest.mark.parametrize('mode,tol', [('fp32', 1e-4), ('fp16', 2e-2)])
def test_standalone_output_block_twenty_classes(monkeypatch, lib, mode, tol):
    monkeypatch.setenv('SEG3D_MODE', mode)
    from segmentation3d.network.module.vnet_outblock import OutputBlock
    g = torch.Generator().manual_seed(0)
    m = OutputBlock(32, 20)
    with torch.no_grad():
        for name, prm in m.named_parameters():
            if name.endswith('gn1.weight') or name.endswith('gn2.weight'):
                prm.copy_(1.0 + 0.3 * torch.randn(prm.shape, generator=g))
            elif name.endswith('.bias'):
                prm.copy_(0.2 * torch.randn(prm.shape, generator=g))
            else:
                prm.copy_(torch.randn(prm.shape, generator=g) * (2.0 / prm[0].numel()) ** 0.5)
        x = torch.randn((2, 32, 8, 8, 16), generator=g)
        sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
        y = F.relu(F.group_norm(F.conv3d(x, sd['conv1.weight'], sd['conv1.bias'], padding=1), 1, sd['gn1.weight'], sd['gn1.bias'], EPS))
        y = F.softmax(F.group_norm(F.conv3d(y, sd['conv2.weight'], sd['conv2.bias']), 1, sd['gn2.weight'], sd['gn2.bias'], EPS), 1)
        got = m.cuda()(x.cuda()).cpu()
    assert got.shape == y.shape == (2, 20, 8, 8, 16)
    err = float((got - y).abs().max())
    print('OutputBlock 20 classes', mode, 'max|dp| %.3g' % err)
    assert err <= tol, (mode, err)
    assert float((got.sum(1) - 1).abs().max()) <= 1e-5
