"""GPU parity tests of the C-ABI kernels against the oracle (run on the B200 box: pytest -m gpu)."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from oracle import net as onet
from oracle.metrics import parity_report

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(scope='module')
def lib():
    from segmentation3d._b200 import lib as L
    L.load()
    assert L.load().seg3d_device_check(0) == 0, L.load().seg3d_last_error()
    return L


def seeded_input(seed, shape, kind='noise'):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g)
    if kind == 'smooth':
        lo = torch.randn((shape[0], shape[1]) + tuple(max(2, s // 8) for s in shape[2:]), generator=g)
        x = torch.nn.functional.interpolate(lo, size=shape[2:], mode='trilinear', align_corners=False) * 2 + 0.3 * x
    return x


def to_ndhwc(x, dtype):   # [N,C,D,H,W] -> [N,D,H,W,C]
    return x.permute(0, 2, 3, 4, 1).contiguous().to(dtype).cuda()


def from_ndhwc(y):
    return y.float().cpu().permute(0, 4, 1, 2, 3).contiguous()


def pack_simt(w, mode, L):
    if mode == L.CONV_T2S2:
        return w.permute(0, 2, 3, 4, 1).reshape(w.shape[0], -1).contiguous().cuda()
    return w.permute(2, 3, 4, 1, 0).reshape(-1, w.shape[1], w.shape[0]).contiguous().cuda()


def pack_tc(w, mode, L, dtype):
    if mode == L.CONV_T2S2:
        return w.permute(2, 3, 4, 1, 0).reshape(-1, w.shape[0]).contiguous().to(dtype).cuda()
    return w.permute(2, 3, 4, 0, 1).reshape(-1, w.shape[0], w.shape[1]).contiguous().to(dtype).cuda()


def run_conv(L, mode, dt, impl, x, w, b, with_stats=True):
    N, Cin, D, H, W = x.shape
    tdt = L.TORCH_DTYPE[dt]
    xd = to_ndhwc(x, tdt)
    if mode == L.CONV_T2S2:
        Cout, od = w.shape[1], (2 * D, 2 * H, 2 * W)
    elif mode == L.CONV_K2S2:
        Cout, od = w.shape[0], (D // 2, H // 2, W // 2)
    else:
        Cout, od = w.shape[0], (D, H, W)
    wp = pack_simt(w, mode, L) if impl == L.IMPL_SIMT else pack_tc(w, mode, L, tdt)
    y = torch.full((N,) + od + (Cout,), float('nan'), dtype=tdt, device='cuda')
    stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    bd = b.cuda() if b is not None else None
    L.call('seg3d_conv3d_fwd', mode, dt, impl, L.ptr(xd), Cin, Cin, L.ptr(wp), L.ptr(bd), L.ptr(y), Cout, Cout,
           N, D, H, W, L.ptr(stats) if with_stats else None, L.stream_ptr())
    torch.cuda.synchronize()
    return from_ndhwc(y), stats.cpu()


def ref_conv(mode, L, x, w, b):
    if mode == L.CONV_K3:
        return F.conv3d(x, w, b, padding=1)
    if mode == L.CONV_K2S2:
        return F.conv3d(x, w, b, stride=2)
    if mode == L.CONV_T2S2:
        return F.conv_transpose3d(x, w, b, stride=2)
    return F.conv3d(x, w, b)


CONV_CASES = [
    # mode name, Cin, Cout, N, D, H, W
    ('K3', 1, 16, 2, 8, 12, 16), ('K3', 16, 32, 1, 6, 10, 8), ('K3', 32, 2, 2, 8, 8, 8), ('K3', 32, 5, 1, 8, 8, 16),
    ('K3', 64, 64, 1, 6, 6, 6), ('K3', 2, 16, 1, 8, 8, 8),
    ('K2S2', 16, 32, 2, 8, 12, 16), ('K2S2', 128, 256, 1, 4, 4, 4),
    ('T2S2', 64, 16, 2, 4, 6, 8), ('T2S2', 256, 128, 1, 2, 2, 2),
    ('K1', 32, 16, 1, 4, 4, 8),
]


@pytest.mark.parametrize('case', CONV_CASES, ids=lambda c: '-'.join(map(str, c)))
def test_conv_simt_fp32_matches_torch(lib, case):
    L = lib
    mname, Cin, Cout, N, D, H, W = case
    mode = getattr(L, 'CONV_' + mname)
    g = torch.Generator().manual_seed(CONV_CASES.index(case))
    x = torch.randn((N, Cin, D, H, W), generator=g)
    wshape = (Cin, Cout, 2, 2, 2) if mode == L.CONV_T2S2 else (Cout, Cin) + {L.CONV_K3: (3, 3, 3), L.CONV_K2S2: (2, 2, 2), L.CONV_K1: (1, 1, 1)}[mode]
    w = torch.randn(wshape, generator=g) * 0.1
    b = torch.randn((Cout,), generator=g) * 0.1
    ref = ref_conv(mode, L, x, w, b)
    y, stats = run_conv(L, mode, L.F32, L.IMPL_SIMT, x, w, b)
    assert y.shape == ref.shape
    assert not torch.isnan(y).any()
    assert (y - ref).abs().max() <= 2e-5 * max(1.0, ref.abs().max())        # fp32 FFMA, different summation order
    # the statistics sum the fp32 values the kernel stores: over thousands of voxels the per-voxel rounding differences
    # from torch add up beyond these bounds, so the sums are taken over the kernel's own output
    s_ref = torch.stack([y.double().flatten(1).sum(1), (y.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats, s_ref, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize('dt_name', ['F16', 'BF16'])
def test_conv_simt_half_storage(lib, dt_name):
    L = lib
    dt = getattr(L, dt_name)
    g = torch.Generator().manual_seed(3)
    x = torch.randn((1, 32, 6, 8, 8), generator=g)
    w = torch.randn((32, 32, 3, 3, 3), generator=g) * 0.05
    xr = x.to(L.TORCH_DTYPE[dt]).float()
    ref = F.conv3d(xr, w, None, padding=1)
    y, _ = run_conv(L, L.CONV_K3, dt, L.IMPL_SIMT, x, w, None)
    tol = 4e-3 if dt == L.F16 else 3e-2
    assert (y - ref).abs().max() <= tol * max(1.0, ref.abs().max())


@pytest.mark.parametrize('dt_name,relu,use_res', [('F32', True, True), ('F32', False, False), ('F16', True, False), ('F16', True, True)])
def test_gn_apply_matches_group_norm(lib, dt_name, relu, use_res):
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    g = torch.Generator().manual_seed(5)
    N, C, D, H, W = 2, 32, 6, 4, 8
    y = torch.randn((N, C, D, H, W), generator=g) * 2 + 0.5
    res = torch.randn((N, C, D, H, W), generator=g)
    gamma, beta = torch.randn(C, generator=g), torch.randn(C, generator=g)
    yq, rq = y.to(tdt).float(), res.to(tdt).float()
    ref = F.group_norm(y, 1, gamma, beta, 1e-5)          # statistics come from the un-rounded fp32 conv results
    mean = y.flatten(1).mean(1).view(N, 1, 1, 1, 1)
    rstd = 1.0 / torch.sqrt(y.flatten(1).var(1, unbiased=False).view(N, 1, 1, 1, 1) + 1e-5)
    ref = (yq - mean) * rstd * gamma.view(1, C, 1, 1, 1) + beta.view(1, C, 1, 1, 1)
    if use_res:
        ref = ref + rq
    if relu:
        ref = F.relu(ref)
    stats = torch.stack([y.double().flatten(1).sum(1), (y.double() ** 2).flatten(1).sum(1)], 1).cuda()
    yd, rd = to_ndhwc(y, tdt), to_ndhwc(res, tdt)
    # write into the second half of a wider (concat) buffer
    out = torch.zeros((N, D, H, W, 2 * C), dtype=tdt, device='cuda')
    gd, bd = gamma.cuda(), beta.cuda()
    L.call('seg3d_gn_apply', dt, L.ptr(yd), C, C, L.ptr(stats), L.ptr(gd), L.ptr(bd), 1e-5,
           L.ptr(rd) if use_res else None, C, L.ptr(out, C), 2 * C, 1 if relu else 0, N, D * H * W, L.stream_ptr())
    torch.cuda.synchronize()
    got = from_ndhwc(out[..., C:])
    assert (out[..., :C] == 0).all()
    tol = 1e-5 if dt == L.F32 else 4e-3
    assert (got - ref).abs().max() <= tol * max(1.0, ref.abs().max())


def _plan_forward(L, sd, x, mode, **kw):
    from segmentation3d._b200.plan import NetPlan
    plan = NetPlan(sd, mode=mode, device='cuda', **kw)
    y = plan.forward(x.cuda()).clone()
    torch.cuda.synchronize()
    return y.cpu()


def test_forward_fp32_matches_golden_and_oracle(lib):
    z = np.load(os.path.join(G, 'forward.npz'))
    meta = json.loads(str(z['meta']))
    for name, arch, cin, cout, wseed, aseed, iseed, shape, kind in meta:
        sd = oinit.init_state_dict(arch, cin, cout, wseed)
        if aseed is not None:
            sd = oinit.randomize_affine(sd, aseed)
        x = seeded_input(iseed, tuple(shape), kind)
        y = _plan_forward(lib, sd, x, 'fp32').numpy()
        gold = z[name]
        d = np.abs(y - gold).max()
        print(name, 'fp32 max|dp| vs reference golden = %.3g' % d)
        assert d <= 1e-3, name                       # BASELINE.json fp32 bar; expected ~1e-5
        assert np.abs(y.sum(1) - 1).max() <= 1e-5


def test_forward_fp32_ties_are_bit_equal(lib):
    """SURVEY D11: ~27% of voxels are exact 0.5/0.5 ties on kaiming-init VNet; they must stay exact."""
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    x = seeded_input(100, (1, 1, 32, 32, 32))
    ref = onet.forward(sd, x)
    y = _plan_forward(lib, sd, x, 'fp32')
    tie_ref = (ref[0, 0] == ref[0, 1])
    tie_new = (y[0, 0] == y[0, 1])
    assert tie_ref.float().mean() > 0.05
    assert (tie_ref == tie_new).float().mean() >= 0.999
    rep = parity_report(ref[0].numpy(), y[0].numpy())
    assert rep['agree'] >= 0.999 and min(rep['dice']) >= 0.999, rep


def _net_forward(arch, cout, sd, x, mode=None):
    """through the plug-in module (segmentation3d.network.<arch>.SegmentationNet), whose default mode is 'auto'"""
    import importlib
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


@pytest.mark.parametrize('arch,cout', [('vnet', 2), ('vbnet', 5)])
def test_forward_default_mode_meets_reduced_precision_bars(lib, arch, cout, monkeypatch):
    """BASELINE.json reduced-precision bars (max|dp| <= 1e-2, label agreement >= 99.9 %, per-class Dice >= 0.999) in the
    mode the plug-in picks by default: fp16 for the binary VNet, the split-operand tensor-core mode for the 5-class VBNet
    (network/_graph.py::resolve_mode - plain fp16 operands measurably miss the rare-class Dice there, next test)."""
    monkeypatch.delenv('SEG3D_MODE', raising=False)
    sd = oinit.init_state_dict(arch, 1, cout, 0)
    x = seeded_input(7, (1, 1, 64, 64, 64), 'smooth')
    ref = onet.forward(sd, x)
    y, mode = _net_forward(arch, cout, sd, x)
    assert mode == ('fp16' if cout <= 2 else 'fp32x')
    rep = parity_report(ref[0].numpy(), y[0].numpy())
    print(arch, 'default mode', mode, rep)
    assert rep['max_abs'] <= 1e-2 and rep['agree'] >= 0.999 and min(rep['dice']) >= 0.999, rep


@pytest.mark.parametrize('arch', ['vnet', 'vbnet'])
@pytest.mark.parametrize('mode,tol', [('fp32', 1e-3), ('fp32x', 1e-3), ('fp16', 1e-2)])
def test_forward_sixteen_classes_like_the_reference_test(lib, arch, mode, tol):
    """The reference's own network test builds a 16-class net (network/vbnet_test.py:9, vnet_test.py): the out-block tail kernels
    are instantiated up to 16 classes and out_block.conv1 runs zero-padded on the generic tensor-core kernel (the folded
    narrow-output kernel takes up to 7).  Probabilities against the oracle in the strict and the reduced modes."""
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, 16, 3), 11)
    x = seeded_input(17, (2, 1, 32, 32, 32), 'smooth')
    ref = onet.forward(sd, x)
    y, resolved = _net_forward(arch, 16, sd, x, mode)
    assert resolved == mode and tuple(y.shape) == (2, 16, 32, 32, 32)
    assert float((y.sum(1) - 1).abs().max()) <= 1e-5
    err = float((y - ref).abs().max())
    print(arch, '16 classes', mode, 'max|dp| %.3g' % err)
    assert err <= tol, (arch, mode, err)
    assert _net_forward(arch, 16, sd, x)[1] == 'fp32x'           # the default mode of a multi-class net


def test_forward_vbnet5_plain_fp16_probability_and_agreement_bars(lib):
    """The explicit fast mode on the 5-class VBNet: max|dp| and label agreement meet the bars.  The per-class Dice of the two
    rare classes (780 and 2107 of 262144 voxels, ~2 % of them within 1e-3 of a tie on random-init weights) is recorded, not
    asserted: oracle/reduced_precision.py reproduces 0.9968-0.9988 for ANY single half-precision rounding source, which is
    why 'auto' does not pick fp16 for multi-class nets."""
    sd = oinit.init_state_dict('vbnet', 1, 5, 0)
    x = seeded_input(7, (1, 1, 64, 64, 64), 'smooth')
    ref = onet.forward(sd, x)
    y = _plan_forward(lib, sd, x, 'fp16')
    rep = parity_report(ref[0].numpy(), y[0].numpy())
    print('vbnet C=5 fp16 (opt-in fast mode)', rep)
    assert rep['max_abs'] <= 1e-2 and rep['agree'] >= 0.999, rep
    assert min(rep['dice'][:3]) >= 0.998 and min(rep['dice']) >= 0.99, rep      # sanity floor only


@pytest.mark.parametrize('arch,cout', [('vnet', 2), ('vbnet', 5)])
def test_forward_bf16_parity_is_recorded(lib, arch, cout):
    """bf16 storage + bf16 tensor-core operands against the fp32 oracle, MEASURED on the GPU (north_star states its bars for
    bf16; SURVEY D9 predicted from a CPU emulation that bf16 misses them on random-init weights, which is why the reduced
    mode is fp16).  The numbers are printed and written to gpurun_out/ for profiles/; asserted is only that bf16 is a sane
    approximation (max|dp| <= 0.1, agreement >= 98 %) and that fp16 is tighter on the same input."""
    sd = oinit.init_state_dict(arch, 1, cout, 0)
    x = seeded_input(7, (1, 1, 64, 64, 64), 'smooth')
    ref = onet.forward(sd, x)
    reps = {m: parity_report(ref[0].numpy(), _plan_forward(lib, sd, x, m)[0].numpy()) for m in ('bf16', 'fp16')}
    print(arch, 'bf16 vs fp16 inference parity on B200', reps)
    out = os.path.join(os.path.dirname(G), '..', 'gpurun_out')
    if os.path.isdir(out):
        with open(os.path.join(out, 'bf16_parity_%s_c%d.json' % (arch, cout)), 'w') as f:
            json.dump({'arch': arch, 'classes': cout, 'input': '64^3 smooth seed 7, kaiming init seed 0', 'bars': 'max_abs<=1e-2, agree>=0.999, dice>=0.999',
                       'bf16': reps['bf16'], 'fp16': reps['fp16']}, f)
    assert reps['bf16']['max_abs'] <= 0.1 and reps['bf16']['agree'] >= 0.98, reps
    assert reps['fp16']['max_abs'] <= reps['bf16']['max_abs']


TC_CASES = [
    # Cin, Cout, N, D, H, W
    (32, 32, 1, 8, 8, 8), (64, 64, 2, 8, 4, 8), (16, 16, 1, 4, 8, 16), (128, 128, 1, 4, 4, 8), (256, 256, 1, 6, 6, 6),
    (32, 64, 1, 12, 12, 12), (64, 16, 1, 16, 16, 16), (256, 64, 2, 2, 6, 10),
]


@pytest.mark.parametrize('dt_name', ['F16', 'BF16'])
@pytest.mark.parametrize('case', TC_CASES, ids=lambda c: '-'.join(map(str, c)))
def test_conv_k3_tcgen05_matches_torch(lib, case, dt_name):
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    Cin, Cout, N, D, H, W = case
    g = torch.Generator().manual_seed(Cin * 7 + Cout)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cout, Cin, 3, 3, 3), generator=g) * (1.0 / (27 * Cin) ** 0.5)
    b = torch.randn((Cout,), generator=g) * 0.1
    xr, wr = x.to(tdt).float(), w.to(tdt).float()          # operands as the tensor core sees them
    ref = F.conv3d(xr.double(), wr.double(), b.double(), padding=1).float()
    y, stats = run_conv(L, L.CONV_K3, dt, L.IMPL_TCGEN05, x, w, b)
    assert not torch.isnan(y).any()
    tol = 2e-3 if dt == L.F16 else 1.6e-2                  # output rounding to the storage type
    err = (y - ref).abs().max()
    assert err <= tol * max(1.0, ref.abs().max()), err
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats, s_ref, rtol=1e-4, atol=1e-2)   # stats are taken before the output rounding


K2_CASES = [(16, 32, 2, 8, 16, 16), (32, 64, 1, 16, 8, 24), (64, 128, 1, 8, 8, 8), (128, 256, 2, 4, 12, 4), (16, 32, 1, 32, 32, 32)]


@pytest.mark.parametrize('case', K2_CASES, ids=lambda c: '-'.join(map(str, c)))
def test_conv_k2s2_tcgen05_matches_torch(lib, case):
    L = lib
    Cin, Cout, N, D, H, W = case
    g = torch.Generator().manual_seed(Cin + Cout)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cout, Cin, 2, 2, 2), generator=g) * (1.0 / (8 * Cin) ** 0.5)
    b = torch.randn((Cout,), generator=g) * 0.1
    ref = F.conv3d(x.half().float().double(), w.half().float().double(), b.double(), stride=2).float()
    y, stats = run_conv(L, L.CONV_K2S2, L.F16, L.IMPL_TCGEN05, x, w, b)
    assert not torch.isnan(y).any()
    assert (y - ref).abs().max() <= 2e-3 * max(1.0, ref.abs().max())
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats, s_ref, rtol=1e-4, atol=1e-2)


T2_CASES = [(64, 16, 1, 8, 8, 8), (128, 32, 2, 4, 8, 8), (256, 64, 1, 4, 4, 8), (256, 128, 1, 6, 6, 6), (64, 16, 1, 16, 16, 16)]


@pytest.mark.parametrize('case', T2_CASES, ids=lambda c: '-'.join(map(str, c)))
def test_conv_t2s2_tcgen05_matches_torch(lib, case):
    L = lib
    Cin, Cout, N, D, H, W = case
    g = torch.Generator().manual_seed(Cin + 3 * Cout)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cin, Cout, 2, 2, 2), generator=g) * (1.0 / Cin ** 0.5)
    b = torch.randn((Cout,), generator=g) * 0.1
    ref = F.conv_transpose3d(x.half().float().double(), w.half().float().double(), b.double(), stride=2).float()
    y, stats = run_conv(L, L.CONV_T2S2, L.F16, L.IMPL_TCGEN05, x, w, b)
    assert not torch.isnan(y).any()
    assert (y - ref).abs().max() <= 2e-3 * max(1.0, ref.abs().max())
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats, s_ref, rtol=1e-4, atol=1e-2)


def test_conv_k2s2_tcgen05_strided_input_view(lib):
    """the down-conv reads the skip half of a concat buffer: channel offset + pitch > Cin"""
    L = lib
    g = torch.Generator().manual_seed(4)
    N, Cin, Cout, D = 1, 16, 32, 16
    x = torch.randn((N, Cin, D, D, D), generator=g)
    w = torch.randn((Cout, Cin, 2, 2, 2), generator=g) * 0.1
    ref = F.conv3d(x.half().float(), w.half().float(), None, stride=2)
    cat = torch.randn((N, D, D, D, 2 * Cin), generator=g).half().cuda()
    cat[..., Cin:] = x.permute(0, 2, 3, 4, 1).half().cuda()
    wp = pack_tc(w, L.CONV_K2S2, L, torch.float16)
    y = torch.empty((N, D // 2, D // 2, D // 2, Cout), dtype=torch.float16, device='cuda')
    L.call('seg3d_conv3d_fwd', L.CONV_K2S2, L.F16, L.IMPL_TCGEN05, L.ptr(cat, Cin), 2 * Cin, Cin, L.ptr(wp), None, L.ptr(y), Cout, Cout,
           N, D, D, D, None, L.stream_ptr())
    torch.cuda.synchronize()
    assert (from_ndhwc(y) - ref).abs().max() <= 2e-3 * max(1.0, ref.abs().max())


def test_forward_fp16_tcgen05_equals_simt_path(lib):
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    x = seeded_input(11, (2, 1, 32, 32, 32), 'smooth')
    a = _plan_forward(lib, sd, x, 'fp16', tc_modes=())
    b = _plan_forward(lib, sd, x, 'fp16')
    ref = onet.forward(sd, x)
    print('simt-vs-tc max', float((a - b).abs().max()), 'tc-vs-oracle', float((b - ref).abs().max()))
    assert (b - ref).abs().max() <= 1e-2
    assert (a - b).abs().max() <= 5e-3


WG_CASES = [
    # mode, Cin, Cout, N, D, H, W
    ('K3', 32, 32, 2, 8, 16, 8), ('K3', 64, 64, 1, 4, 16, 16), ('K3', 16, 16, 1, 8, 8, 8), ('K3', 128, 128, 1, 4, 12, 12),
    ('K3', 256, 256, 2, 2, 6, 6), ('K3', 32, 16, 1, 8, 16, 16), ('K3', 16, 64, 1, 4, 8, 8), ('K3', 1, 16, 1, 8, 8, 8),
    ('K2S2', 16, 32, 1, 8, 8, 8), ('T2S2', 64, 16, 1, 4, 4, 8),
    ('K3', 64, 32, 1, 4, 24, 8), ('K3', 16, 32, 2, 5, 16, 16), ('K3', 64, 16, 1, 4, 16, 8), ('K3', 32, 32, 1, 3, 40, 24),   # nine-taps-per-MMA path
    ('K2S2', 32, 64, 2, 8, 32, 16), ('K2S2', 64, 128, 1, 4, 16, 16), ('K2S2', 128, 256, 1, 4, 12, 12),
    ('T2S2', 128, 32, 2, 4, 16, 8), ('T2S2', 256, 64, 1, 2, 12, 12), ('T2S2', 256, 128, 1, 2, 6, 6),
    # x = the upper half of a 2*Cin-wide buffer, as every down conv reads its skip input from the concat buffer
    ('K2S2', 16, 32, 2, 8, 12, 16, 'upper'), ('K2S2', 64, 128, 1, 8, 8, 8, 'upper'), ('K3', 32, 32, 2, 8, 16, 8, 'upper'),
    # out_block.conv1 on the tensor cores: Cout padded to 16, only the first 2 / 5 dy channels nonzero
    ('K3', 32, 16, 2, 8, 16, 8, 'dy2'), ('K3', 32, 16, 1, 6, 24, 16, 'dy5'),
]


@pytest.mark.parametrize('dt_name', ['F32', 'BF16'])
@pytest.mark.parametrize('case', WG_CASES, ids=lambda c: '-'.join(map(str, c)))
def test_conv_wgrad_matches_torch(lib, case, dt_name):
    """seg3d_conv3d_wgrad against float64 autograd: |got - ref| <= 2e-5 sum |x| |dy| per weight (fp32 accumulation)"""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    mname, Cin, Cout, N, D, H, W = case[:7]
    variant = case[7] if len(case) > 7 else ''
    mode = getattr(L, 'CONV_' + mname)
    g = torch.Generator().manual_seed(Cin + 5 * Cout)
    x = torch.randn((N, Cin, D, H, W), generator=g).to(tdt).float()
    if mode == L.CONV_T2S2:
        wshape, od = (Cin, Cout, 2, 2, 2), (2 * D, 2 * H, 2 * W)
    elif mode == L.CONV_K2S2:
        wshape, od = (Cout, Cin, 2, 2, 2), (D // 2, H // 2, W // 2)
    else:
        wshape, od = (Cout, Cin, 3, 3, 3), (D, H, W)
    dy = torch.randn((N, Cout) + od, generator=g).to(tdt).float()
    if variant.startswith('dy'):
        dy[:, int(variant[2:]):] = 0
    w = torch.zeros(wshape, dtype=torch.float64, requires_grad=True)
    y = ref_conv(mode, L, x.double(), w, None)
    (y * dy.double()).sum().backward()
    ref = w.grad
    wa = torch.zeros(wshape, dtype=torch.float64, requires_grad=True)
    ya = ref_conv(mode, L, x.double().abs(), wa, None)
    (ya * dy.double().abs()).sum().backward()
    mag = wa.grad
    xd, dyd = to_ndhwc(x, tdt), to_ndhwc(dy, tdt)
    x_ld, x_off = Cin, 0
    if variant == 'upper':
        wide = (torch.randn(xd.shape[:-1] + (2 * Cin,), generator=g) * 1e3).to(tdt).cuda()      # the lower half must not be read
        wide[..., Cin:] = xd
        xd, x_ld, x_off = wide, 2 * Cin, Cin
    taps = 27 if mode == L.CONV_K3 else 8
    dw = torch.zeros((taps * Cin * Cout,), dtype=torch.float32, device='cuda')
    L.call('seg3d_conv3d_wgrad', mode, dt, L.ptr(xd, x_off), x_ld, Cin, L.ptr(dyd), Cout, Cout, L.ptr(dw), N, D, H, W, L.stream_ptr())
    torch.cuda.synchronize()
    if mode == L.CONV_T2S2:
        got = dw.view(Cin, 2, 2, 2, Cout).permute(0, 4, 1, 2, 3).cpu()
    else:
        k = 3 if mode == L.CONV_K3 else 2
        got = dw.view(k, k, k, Cin, Cout).permute(4, 3, 0, 1, 2).cpu()
    err = (got.double() - ref).abs()
    assert bool((err <= 2e-5 * mag).all()), float((err / (mag + 1e-300)).max())
    if variant.startswith('dy'):
        assert bool((got[int(variant[2:]):] == 0).all()), 'gradient of an all-zero dy channel'


def test_forward_batch_equals_single(lib):
    sd = oinit.init_state_dict('vnet', 1, 2, 1)
    x = seeded_input(9, (3, 1, 16, 32, 16))
    yb = _plan_forward(lib, sd, x, 'fp32')
    y0 = _plan_forward(lib, sd, x[1:2], 'fp32')
    assert (yb[1:2] - y0).abs().max() <= 1e-6     # GroupNorm is per sample: batching must not change results


NARROW_CASES = [
    # Cin, Cout, N, D, H, W  (H not a multiple of the 10-row tile, D shorter/longer than a z segment)
    (32, 2, 2, 16, 16, 16), (32, 5, 1, 8, 24, 8), (16, 3, 1, 5, 10, 16), (64, 2, 1, 12, 32, 8), (32, 7, 3, 32, 48, 48),
]


@pytest.mark.parametrize('case', NARROW_CASES, ids=lambda c: '-'.join(map(str, c)))
@pytest.mark.parametrize('dt_name', ['F16', 'BF16'])
def test_conv_k3_narrow_matches_torch(lib, case, dt_name):
    """seg3d_conv3d_k3_narrow_fwd (taps folded into N, epilogue gather) vs F.conv3d on the same rounded operands."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    Cin, C, N, D, H, W = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn((N, Cin, D, H, W), generator=g).to(tdt).float()
    w = (torch.randn((C, Cin, 3, 3, 3), generator=g) * 0.1).to(tdt).float()
    b = torch.randn((C,), generator=g) * 0.1
    ref = F.conv3d(x, w, b, padding=1)
    NP = L.load().seg3d_conv3d_k3_narrow_np(C)
    assert NP % 16 == 0 and NP >= 9 * C
    wf = torch.zeros((3, NP, Cin))
    wf[:, :9 * C] = w.permute(2, 3, 4, 0, 1).reshape(3, 9 * C, Cin)
    wf = wf.to(tdt).cuda()
    xd = to_ndhwc(x, tdt)
    y = torch.full((N, D, H, W, C), float('nan'), dtype=torch.float32, device='cuda')
    stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    L.call('seg3d_conv3d_k3_narrow_fwd', dt, L.ptr(xd), Cin, Cin, L.ptr(wf), L.ptr(b.cuda()), L.ptr(y), C,
           N, D, H, W, L.ptr(stats), L.stream_ptr())
    torch.cuda.synchronize()
    yc = from_ndhwc(y)
    assert not torch.isnan(yc).any()
    assert (yc - ref).abs().max() <= 2e-4 * max(1.0, float(ref.abs().max()))     # fp32 accumulate, different order
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats.cpu(), s_ref, rtol=1e-4, atol=1e-2)


@pytest.mark.parametrize('shape', [(2, 8, 12, 16), (1, 20, 32, 24), (3, 5, 16, 8), (1, 96, 96, 96)], ids=str)
@pytest.mark.parametrize('dt_name', ['F16', 'BF16'])
def test_conv_cin1_tensor_core_matches_torch(lib, shape, dt_name):
    """Input block on the tensor cores (im2col tile built in shared memory, hi/lo weight split): IMPL_AUTO vs F.conv3d
    with the input rounded to the storage type and the weights left in fp32."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, D, H, W = shape
    g = torch.Generator().manual_seed(D * 7 + W)
    x = torch.randn((N, 1, D, H, W), generator=g).to(tdt).float()
    w = torch.randn((16, 1, 3, 3, 3), generator=g) * 0.3
    b = torch.randn((16,), generator=g) * 0.1
    ref = F.conv3d(x, w, b, padding=1)
    ld = 32                                            # written into the upper half of a 32-channel concat buffer
    y = torch.full((N, D, H, W, ld), float('nan'), dtype=tdt, device='cuda')
    stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    xd = x.reshape(N, D, H, W).to(tdt).cuda()
    wp = pack_simt(w, L.CONV_K3, L)
    L.call('seg3d_conv3d_fwd', L.CONV_K3, dt, L.IMPL_AUTO, L.ptr(xd), 1, 1, L.ptr(wp), L.ptr(b.cuda()), L.ptr(y, 16), ld, 16,
           N, D, H, W, L.ptr(stats), L.stream_ptr())
    torch.cuda.synchronize()
    assert torch.isnan(y[..., :16].float()).all()      # the other half of the concat buffer is untouched
    yc = from_ndhwc(y[..., 16:])
    assert not torch.isnan(yc).any()
    tol_store = 2.0 ** (-11 if dt == L.F16 else -8)    # output rounding to the storage type
    assert (yc - ref).abs().max() <= tol_store * float(ref.abs().max()) * 1.01 + 1e-5
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    rt = 1e-5 if dt == L.F16 else 2e-4                 # the sums come from the fp32 accumulators (hi+lo weights)
    assert torch.allclose(stats.cpu(), s_ref, rtol=rt, atol=rt * float(s_ref[:, 1].max()))


@pytest.mark.parametrize('shape', [(2, 8, 12, 16), (1, 20, 40, 24), (3, 5, 16, 8), (2, 33, 70, 72), (1, 96, 96, 96)], ids=str)
@pytest.mark.parametrize('dt_name,lo', [('F16', 0), ('BF16', 0), ('F16', 1)])
def test_conv_cin1_toeplitz_matches_torch(lib, monkeypatch, shape, dt_name, lo):
    """Input block as a TMA-fed banded-Toeplitz GEMM (seg3d_conv3d_cin1_fwd, row-padded input): the three epilogue modes vs
    F.conv3d / F.group_norm on the input rounded to the storage type with fp32 weights.  Shapes cover partial 32 x 32 tiles,
    several z segments and W / 8 not a multiple of the 4-segment box."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, D, H, W = shape
    monkeypatch.setenv('SEG3D_CIN1_LO', str(lo))       # 0 (default): weights rounded to the storage type; 1: hi + lo split, fp32-accurate
    g = torch.Generator().manual_seed(D * 7 + W)
    x = torch.randn((N, 1, D, H, W), generator=g).to(tdt).float()
    w = torch.randn((16, 1, 3, 3, 3), generator=g) * 0.3
    b = torch.randn((16,), generator=g) * 0.1
    gamma = torch.rand((16,), generator=g) + 0.5
    beta = torch.randn((16,), generator=g) * 0.2
    w_seen = w if lo else w.to(tdt).float()
    ref = F.conv3d(x, w_seen, b, padding=1)
    ref_gn = F.relu(F.group_norm(ref, 1, gamma, beta, 1e-5))
    pitch = W + L.CIN1_PAD
    xp = torch.zeros((N, D, H, pitch), dtype=tdt, device='cuda')
    xp[..., L.CIN1_LEFT:L.CIN1_LEFT + W] = x[:, 0].to(tdt).cuda()
    wp = pack_simt(w, L.CONV_K3, L)
    bd, gd, btd = b.cuda(), gamma.cuda(), beta.cuda()
    ld = 32                                            # written into the upper half of a 32-channel concat buffer
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    rt = 1e-5 if dt == L.F16 else 2e-4                 # the sums come from the fp32 accumulators (hi+lo weights)
    tol_store = 2.0 ** (-11 if dt == L.F16 else -8)    # output rounding to the storage type

    def run(epi, stats):
        y = torch.full((N, D, H, W, ld), float('nan'), dtype=tdt, device='cuda')
        L.call('seg3d_conv3d_cin1_fwd', dt, epi, L.ptr(xp), pitch, L.ptr(wp), L.ptr(bd), None if epi == 1 else L.ptr(y, 16), ld,
               N, D, H, W, L.ptr(stats), L.ptr(gd), L.ptr(btd), 1e-5, L.stream_ptr())
        torch.cuda.synchronize()
        return y

    # mode 0: raw conv + sums
    st0 = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    y0 = run(0, st0)
    assert torch.isnan(y0[..., :16].float()).all()     # the other half of the concat buffer is untouched
    yc = from_ndhwc(y0[..., 16:])
    assert not torch.isnan(yc).any()
    assert (yc - ref).abs().max() <= tol_store * float(ref.abs().max()) * 1.01 + 1e-5
    assert torch.allclose(st0.cpu(), s_ref, rtol=rt, atol=rt * float(s_ref[:, 1].max()))
    # mode 1: the same sums, bit for bit, nothing stored
    st1 = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    run(1, st1)
    assert torch.allclose(st1.cpu(), s_ref, rtol=rt, atol=rt * float(s_ref[:, 1].max()))
    # mode 2: relu(GroupNorm(conv)) from the finished sums
    y2 = run(2, st1)
    assert torch.isnan(y2[..., :16].float()).all()
    yg = from_ndhwc(y2[..., 16:])
    assert not torch.isnan(yg).any()
    assert (yg - ref_gn).abs().max() <= tol_store * float(ref_gn.abs().max()) * 1.01 + 2e-5


@pytest.mark.parametrize('shape', [(2, 8, 12, 16), (1, 20, 40, 24), (2, 33, 70, 72), (2, 96, 96, 96)], ids=str)
@pytest.mark.parametrize('dt_name', ['BF16', 'F16'])
def test_wgrad_cin1_toeplitz_matches_torch(lib, shape, dt_name):
    """Weight gradient of the input block with the Toeplitz operands (seg3d_conv3d_cin1_wgrad: MN-major dy segments and padded
    input windows, K = segments) vs the float64 gradient of F.conv3d on the same stored (rounded) tensors."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, D, H, W = shape
    g = torch.Generator().manual_seed(D * 11 + W)
    x = torch.randn((N, 1, D, H, W), generator=g).to(tdt)
    dy = (torch.randn((N, 16, D, H, W), generator=g) * 0.05).to(tdt)
    w = torch.zeros((16, 1, 3, 3, 3), dtype=torch.float64, requires_grad=True)
    F.conv3d(x.double(), w, None, padding=1).backward(dy.double())
    ref = w.grad.permute(2, 3, 4, 1, 0).reshape(27, 16)                  # [tap][co]
    pitch = W + L.CIN1_PAD
    xp = torch.zeros((N, D, H, pitch), dtype=tdt, device='cuda')
    xp[..., L.CIN1_LEFT:L.CIN1_LEFT + W] = x[:, 0].cuda()
    dyd = dy.permute(0, 2, 3, 4, 1).contiguous().cuda()
    dw = torch.zeros((27, 16), dtype=torch.float32, device='cuda')
    L.call('seg3d_conv3d_cin1_wgrad', dt, L.ptr(xp), pitch, L.ptr(dyd), 16, L.ptr(dw), N, D, H, W, L.stream_ptr())
    L.call('seg3d_conv3d_cin1_wgrad', dt, L.ptr(xp), pitch, L.ptr(dyd), 16, L.ptr(dw), N, D, H, W, L.stream_ptr())   # accumulates
    torch.cuda.synchronize()
    got = dw.cpu().double() / 2
    scale = float(ref.abs().max())
    assert float((got - ref).abs().max()) <= 2e-4 * scale + 1e-6, (float((got - ref).abs().max()), scale)


@pytest.mark.parametrize('case', [('K2S2', 16, 32, 2, 8, 12, 16), ('K2S2', 64, 128, 1, 8, 8, 8), ('T2S2', 64, 16, 2, 4, 6, 8),
                                  ('T2S2', 256, 128, 1, 2, 4, 4)], ids=lambda c: '-'.join(map(str, c)))
def test_conv_gn_relu_two_pass_matches_torch(lib, case):
    """seg3d_conv3d_gn_relu_fwd (statistics pass, then GroupNorm + ReLU in the epilogue) vs relu(group_norm(conv)) in fp32
    on the same fp16-rounded operands; the output lands in one half of a wider concat buffer."""
    L = lib
    dt, tdt = L.F16, torch.float16
    mname, Cin, Cout, N, D, H, W = case
    mode = getattr(L, 'CONV_' + mname)
    g = torch.Generator().manual_seed(Cin + Cout)
    x = torch.randn((N, Cin, D, H, W), generator=g).to(tdt).float()
    wshape = (Cin, Cout, 2, 2, 2) if mode == L.CONV_T2S2 else (Cout, Cin, 2, 2, 2)
    w = (torch.randn(wshape, generator=g) * 0.1).to(tdt).float()
    b = torch.randn((Cout,), generator=g) * 0.1
    gamma = torch.rand((Cout,), generator=g) + 0.5
    beta = torch.randn((Cout,), generator=g) * 0.2
    ref = F.relu(F.group_norm(ref_conv(mode, L, x, w, b), 1, gamma, beta, 1e-5))
    od = ref.shape[2:]
    ld = 2 * Cout
    y = torch.full((N,) + tuple(od) + (ld,), float('nan'), dtype=tdt, device='cuda')
    stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    xd, wp = to_ndhwc(x, tdt), pack_tc(w, mode, L, tdt)
    bd, gd, btd = b.cuda(), gamma.cuda(), beta.cuda()
    for ps in (0, 1):
        L.call('seg3d_conv3d_gn_relu_fwd', mode, dt, ps, L.ptr(xd), Cin, Cin, L.ptr(wp), L.ptr(bd), L.ptr(y, Cout), ld, Cout,
               N, D, H, W, L.ptr(stats), L.ptr(gd), L.ptr(btd), 1e-5, L.stream_ptr())
        torch.cuda.synchronize()
        if ps == 0:
            assert torch.isnan(y.float()).all()                     # the statistics pass stores nothing
    assert torch.isnan(y[..., :Cout].float()).all()
    yc = from_ndhwc(y[..., Cout:])
    assert (yc - ref).abs().max() <= 2.0 ** -10 * max(1.0, float(ref.abs().max())) + 1e-4


@pytest.mark.parametrize('shape', [(2, 16, 16, 16), (1, 8, 24, 8), (3, 32, 48, 48)], ids=str)
@pytest.mark.parametrize('dt_name', ['F16', 'BF16'])
def test_conv_k3_narrow_fused_gn_residual_equals_unfused(lib, shape, dt_name):
    """seg3d_conv3d_k3_narrow_gn_fwd (GroupNorm + residual + ReLU formed in shared memory) must reproduce seg3d_gn_apply
    followed by seg3d_conv3d_k3_narrow_fwd: the operand rounding point and the convolution are the same."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, D, H, W = shape
    Cin, C = 32, 2
    g = torch.Generator().manual_seed(N * 100 + W)
    raw = to_ndhwc(torch.randn((N, Cin, D, H, W), generator=g) * 2.0 + 0.3, tdt)
    res = torch.full((N, D, H, W, 2 * Cin), float('nan'), dtype=tdt, device='cuda')     # residual = one half of a wider buffer
    res[..., Cin:] = to_ndhwc(torch.randn((N, Cin, D, H, W), generator=g), tdt)
    gamma = (torch.rand((Cin,), generator=g) + 0.5).cuda()
    beta = (torch.randn((Cin,), generator=g) * 0.2).cuda()
    w = (torch.randn((C, Cin, 3, 3, 3), generator=g) * 0.1)
    b = (torch.randn((C,), generator=g) * 0.1).cuda()
    NP = L.load().seg3d_conv3d_k3_narrow_np(C)
    wf = torch.zeros((3, NP, Cin))
    wf[:, :9 * C] = w.permute(2, 3, 4, 0, 1).reshape(3, 9 * C, Cin)
    wf = wf.to(tdt).cuda()
    rf = raw.float()
    gstats = torch.stack([rf.double().flatten(1).sum(1), (rf.double() ** 2).flatten(1).sum(1)], 1).contiguous()
    nvox = D * H * W
    # unfused: gn_apply (+res, relu) -> narrow conv
    act = torch.empty((N, D, H, W, Cin), dtype=tdt, device='cuda')
    L.call('seg3d_gn_apply', dt, L.ptr(raw), Cin, Cin, L.ptr(gstats), L.ptr(gamma), L.ptr(beta), 1e-5, L.ptr(res, Cin), 2 * Cin,
           L.ptr(act), Cin, 1, N, nvox, L.stream_ptr())
    y0 = torch.full((N, D, H, W, C), float('nan'), dtype=torch.float32, device='cuda')
    s0 = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    L.call('seg3d_conv3d_k3_narrow_fwd', dt, L.ptr(act), Cin, Cin, L.ptr(wf), L.ptr(b), L.ptr(y0), C, N, D, H, W, L.ptr(s0), L.stream_ptr())
    # fused
    y1 = torch.full((N, D, H, W, C), float('nan'), dtype=torch.float32, device='cuda')
    s1 = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    L.call('seg3d_conv3d_k3_narrow_gn_fwd', dt, L.ptr(raw), Cin, L.ptr(res, Cin), 2 * Cin, Cin, L.ptr(gstats), L.ptr(gamma), L.ptr(beta),
           1e-5, L.ptr(wf), L.ptr(b), L.ptr(y1), C, N, D, H, W, L.ptr(s1), L.stream_ptr())
    torch.cuda.synchronize()
    assert not torch.isnan(y1).any()
    assert torch.equal(y0, y1)
    assert torch.allclose(s0, s1, rtol=1e-9, atol=1e-6)


@pytest.mark.parametrize('shape', [(2, 16, 16, 16), (1, 8, 24, 8), (2, 20, 40, 24), (3, 32, 48, 48)], ids=str)
@pytest.mark.parametrize('dt_name', ['F16', 'BF16'])
def test_up_block_gn_folded_into_both_consumers_equals_unfused(lib, shape, dt_name):
    """The last up-block with up_gn's apply pass folded into its two readers: seg3d_conv3d_k3_gnin_fwd (z-march kernel with the
    transform stage) and seg3d_conv3d_k3_narrow_gn2_fwd (fused out-block convolution whose residual's lower half is still raw)
    must reproduce seg3d_gn_apply -> seg3d_conv3d_fwd -> seg3d_conv3d_k3_narrow_gn_fwd bit for bit."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, D, H, W = shape
    g = torch.Generator().manual_seed(N * 7 + W)
    nvox = D * H * W
    raw_up = to_ndhwc(torch.randn((N, 16, D, H, W), generator=g) * 1.5 + 0.2, tdt)            # raw result of the transposed conv
    skip = to_ndhwc(torch.relu(torch.randn((N, 16, D, H, W), generator=g)), tdt)
    gam_u = (torch.rand((16,), generator=g) + 0.5).cuda()
    bet_u = (torch.randn((16,), generator=g) * 0.2).cuda()
    st_u = torch.stack([raw_up.double().flatten(1).sum(1), (raw_up.double() ** 2).flatten(1).sum(1)], 1).contiguous()
    w = (torch.randn((32, 32, 3, 3, 3), generator=g) * 0.06).to(tdt).float()
    b = (torch.randn((32,), generator=g) * 0.1).cuda()
    wp = pack_tc(w, L.CONV_K3, L, tdt)
    gam_r = (torch.rand((32,), generator=g) + 0.5).cuda()
    bet_r = (torch.randn((32,), generator=g) * 0.2).cuda()
    C = 2
    w1 = torch.randn((C, 32, 3, 3, 3), generator=g) * 0.1
    b1 = (torch.randn((C,), generator=g) * 0.1).cuda()
    NP = L.load().seg3d_conv3d_k3_narrow_np(C)
    wf = torch.zeros((3, NP, 32))
    wf[:, :9 * C] = w1.permute(2, 3, 4, 0, 1).reshape(3, 9 * C, 32)
    wf = wf.to(tdt).cuda()

    def run(fused):
        cat = torch.empty((N, D, H, W, 32), dtype=tdt, device='cuda')
        cat[..., 16:] = skip
        raw2 = torch.full((N, D, H, W, 32), float('nan'), dtype=tdt, device='cuda')
        st2 = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
        y = torch.full((N, D, H, W, C), float('nan'), dtype=torch.float32, device='cuda')
        st3 = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
        if fused:
            cat[..., :16] = raw_up                   # the lower half stays raw
            L.call('seg3d_conv3d_k3_gnin_fwd', dt, L.ptr(cat), 32, 32, 16, L.ptr(st_u), L.ptr(gam_u), L.ptr(bet_u), 1e-5, L.ptr(wp),
                   L.ptr(b), L.ptr(raw2), 32, 32, N, D, H, W, L.ptr(st2), L.stream_ptr())
            L.call('seg3d_conv3d_k3_narrow_gn2_fwd', dt, L.ptr(raw2), 32, L.ptr(cat), 32, 32, L.ptr(st2), L.ptr(gam_r), L.ptr(bet_r), 1e-5,
                   16, L.ptr(st_u), L.ptr(gam_u), L.ptr(bet_u), L.ptr(wf), L.ptr(b1), L.ptr(y), C, N, D, H, W, L.ptr(st3), L.stream_ptr())
        else:
            L.call('seg3d_gn_apply', dt, L.ptr(raw_up), 16, 16, L.ptr(st_u), L.ptr(gam_u), L.ptr(bet_u), 1e-5, None, 0,
                   L.ptr(cat), 32, 1, N, nvox, L.stream_ptr())
            L.call('seg3d_conv3d_fwd', L.CONV_K3, dt, L.IMPL_TCGEN05, L.ptr(cat), 32, 32, L.ptr(wp), L.ptr(b), L.ptr(raw2), 32, 32,
                   N, D, H, W, L.ptr(st2), L.stream_ptr())
            L.call('seg3d_conv3d_k3_narrow_gn_fwd', dt, L.ptr(raw2), 32, L.ptr(cat), 32, 32, L.ptr(st2), L.ptr(gam_r), L.ptr(bet_r), 1e-5,
                   L.ptr(wf), L.ptr(b1), L.ptr(y), C, N, D, H, W, L.ptr(st3), L.stream_ptr())
        torch.cuda.synchronize()
        return raw2, st2, y, st3

    r0, s0, y0, t0 = run(False)
    r1, s1, y1, t1 = run(True)
    assert not torch.isnan(r1.float()).any() and not torch.isnan(y1).any()
    assert torch.equal(r0, r1)
    assert torch.allclose(s0, s1, rtol=1e-9, atol=1e-6)
    assert torch.equal(y0, y1)
    assert torch.allclose(t0, t1, rtol=1e-9, atol=1e-6)


def _split_rows(x5):
    """[N,C,D,H,W] fp32 -> NDHWC rows [hi(C) | lo(C)] f16 on the GPU, and the value the kernels see (hi + lo)"""
    rows = x5.permute(0, 2, 3, 4, 1).contiguous()
    hi = rows.half()
    lo = (rows - hi.float()).half()
    seen = (hi.float() + lo.float()).permute(0, 4, 1, 2, 3).contiguous()
    return torch.cat([hi, lo], dim=-1).contiguous().cuda(), seen


@pytest.mark.parametrize('case', [(32, 32, 2, 8, 18, 16), (16, 16, 1, 12, 40, 24), (32, 32, 1, 5, 16, 8), (16, 64, 2, 6, 20, 8)],
                         ids=lambda c: '-'.join(map(str, c)))
def test_conv_k3_split_zmarch_matches_torch(lib, case):
    """seg3d_conv3d_split_fwd on rows [hi(Cin) | lo(Cin)] (the z-march kernel with the three-product k loop for Cin = 16 / 32):
    fp32 result within 2e-5 of F.conv3d in fp32 on the values the kernel sees; sums from the fp32 accumulators."""
    L = lib
    Cin, Cout, N, D, H, W = case
    g = torch.Generator().manual_seed(Cin * 3 + Cout + D)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cout, Cin, 3, 3, 3), generator=g) * 0.1
    b = torch.randn((Cout,), generator=g) * 0.1
    xd, xs = _split_rows(x)
    q = w.permute(2, 3, 4, 0, 1).reshape(27, Cout, Cin)
    whi = q.half()
    wlo = (q - whi.float()).half()
    wp = torch.cat([whi, wlo], dim=-1).contiguous().cuda()
    wseen = (whi.float() + wlo.float()).view(3, 3, 3, Cout, Cin).permute(3, 4, 0, 1, 2).contiguous()
    ref = F.conv3d(xs.double(), wseen.double(), b.double(), padding=1).float()
    y = torch.full((N, D, H, W, Cout), float('nan'), dtype=torch.float32, device='cuda')
    stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    L.call('seg3d_conv3d_split_fwd', L.CONV_K3, L.ptr(xd), 2 * Cin, Cin, Cin, L.ptr(wp), L.ptr(b.cuda()), L.ptr(y), Cout, Cout,
           N, D, H, W, L.ptr(stats), L.stream_ptr())
    torch.cuda.synchronize()
    yc = y.cpu().permute(0, 4, 1, 2, 3)
    assert not torch.isnan(yc).any()
    assert float((yc - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats.cpu(), s_ref, rtol=1e-5, atol=1e-5 * float(s_ref[:, 1].max()))


@pytest.mark.parametrize('case', [(2, 2, 8, 20, 16), (5, 1, 12, 18, 24), (3, 1, 5, 10, 8)], ids=lambda c: '-'.join(map(str, c)))
def test_conv_narrow_split_matches_torch(lib, case):
    """seg3d_conv3d_k3_narrow_split_fwd (out_block.conv1 in the strict mode: folded in-plane taps on split operands)."""
    L = lib
    C, N, D, H, W = case
    Cin = 32
    g = torch.Generator().manual_seed(C * 5 + D)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((C, Cin, 3, 3, 3), generator=g) * 0.1
    b = torch.randn((C,), generator=g) * 0.1
    xd, xs = _split_rows(x)
    NP = L.load().seg3d_conv3d_k3_narrow_np(C)
    wf = torch.zeros((3, NP, Cin))
    wf[:, :9 * C] = w.permute(2, 3, 4, 0, 1).reshape(3, 9 * C, Cin)
    fhi = wf.half()
    flo = (wf - fhi.float()).half()
    wp = torch.cat([fhi, flo], dim=-1).contiguous().cuda()
    wseen = (fhi.float() + flo.float())[:, :9 * C].view(3, 3, 3, C, Cin).permute(3, 4, 0, 1, 2).contiguous()
    ref = F.conv3d(xs.double(), wseen.double(), b.double(), padding=1).float()
    y = torch.full((N, D, H, W, C), float('nan'), dtype=torch.float32, device='cuda')
    stats = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    L.call('seg3d_conv3d_k3_narrow_split_fwd', L.ptr(xd), 2 * Cin, Cin, L.ptr(wp), L.ptr(b.cuda()), L.ptr(y), C, N, D, H, W,
           L.ptr(stats), L.stream_ptr())
    torch.cuda.synchronize()
    yc = y.cpu().permute(0, 4, 1, 2, 3)
    assert not torch.isnan(yc).any()
    assert float((yc - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
    s_ref = torch.stack([ref.double().flatten(1).sum(1), (ref.double() ** 2).flatten(1).sum(1)], 1)
    assert torch.allclose(stats.cpu(), s_ref, rtol=1e-5, atol=1e-5 * float(s_ref[:, 1].max()))


@pytest.mark.parametrize('arch,cout,seed', [('vnet', 2, 0), ('vbnet', 5, 1)])
def test_forward_split_operand_strict_mode_on_tensor_cores(lib, arch, cout, seed):
    """mode 'fp32x': f16 hi/lo split operands, three MMAs per product, fp32 raw tensors.  Must meet the STRICT bar
    (max |dp| <= 1e-3, north_star fp32/TF32 mode) - and in fact lands within 1e-4 of the fp32 oracle - for both networks,
    including the VBNet 5-class case whose rare-class Dice misses 0.999 in plain fp16."""
    sd = oinit.init_state_dict(arch, 1, cout, seed)
    x = seeded_input(40 + seed, (1, 1, 64, 64, 64), 'smooth')
    ref = onet.forward(sd, x)
    y = _plan_forward(lib, sd, x, 'fp32x')
    rep = parity_report(ref[0].numpy(), y[0].numpy())
    print(arch, 'fp32x', rep)
    assert rep['max_abs'] <= 1e-4, rep
    assert rep['agree'] >= 0.9999 and min(rep['dice']) >= 0.9999, rep


def test_forward_cuda_graph_replay_equals_eager(lib):
    """SEG3D_GRAPH=1: the captured forward must reproduce the eager one bit for bit, also after the weights changed in place."""
    from segmentation3d._b200.plan import NetPlan
    sd = oinit.init_state_dict('vnet', 1, 2, 2)
    x = seeded_input(12, (1, 1, 32, 32, 32)).cuda()
    eager = NetPlan(sd, mode='fp16', device='cuda')
    graph = NetPlan(sd, mode='fp16', device='cuda')
    graph.use_graph = True
    y0 = eager.forward(x).clone()
    y1 = graph.forward(x).clone()          # eager warm-up + capture + replay
    y2 = graph.forward(x).clone()          # replay only
    assert torch.equal(y0, y1) and torch.equal(y0, y2)
    sd2 = {k: (v * 1.01 if v.dim() == 5 else v) for k, v in sd.items()}
    eager.refresh(sd2); graph.refresh(sd2)
    assert torch.equal(eager.forward(x), graph.forward(x))
    x2 = seeded_input(13, (1, 1, 32, 32, 32)).cuda()
    assert torch.equal(eager.forward(x2), graph.forward(x2))


@pytest.mark.parametrize('dt_name', ['F32', 'BF16', 'F16'])
@pytest.mark.parametrize('C,nvox,two_grads,use_res,remask', [(32, 1000, True, True, False), (16, 517, False, False, False), (64, 96, True, False, False),
                                                             (256, 40, False, True, False), (16, 517, False, False, True), (64, 96, True, False, True),
                                                             (32, 4001, False, False, True)],
                         ids=['c32', 'c16', 'c64', 'c256', 'c16-remask', 'c64-remask', 'c32-remask'])
def test_gn_bwd_matches_closed_form(lib, dt_name, C, nvox, two_grads, use_res, remask):
    """seg3d_gn_bwd (both passes) against the closed-form GroupNorm(1,C)+ReLU(+residual) backward in float64, on the
    same stored (rounded) tensors: dy, dres, dgamma, dbeta, dbias and the per-sample sums.  remask: out = NULL, the ReLU mask
    is recomputed from the stored raw tensor (units without a residual)."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, eps = 2, 1e-5
    g = torch.Generator().manual_seed(C + nvox)
    q = lambda t: t.to(tdt).cuda()                                  # noqa: E731  (stored tensors)
    y = q(torch.randn((N, nvox, C), generator=g) * 1.5 + 0.3)
    res = q(torch.randn((N, nvox, C), generator=g))
    gamma, beta = torch.randn(C, generator=g).cuda() + 1.0, torch.randn(C, generator=g).cuda() * 0.3
    g0w = q(torch.randn((N, nvox, 2 * C), generator=g) * 1e-3)       # contribution 0 lives in the upper half of a 2C-wide buffer
    g1 = q(torch.randn((N, nvox, C), generator=g) * 1e-3)
    yd = y.double()
    cnt = float(nvox * C)
    stats = torch.stack([yd.flatten(1).sum(1), (yd * yd).flatten(1).sum(1)], 1).contiguous()
    mean = (stats[:, 0] / cnt).view(N, 1, 1)
    var = (stats[:, 1] / cnt).view(N, 1, 1) - mean * mean
    rstd = 1.0 / torch.sqrt(var + eps)
    xhat = (yd - mean) * rstd
    z = xhat * gamma.double() + beta.double() + (res.double() if use_res else 0.0)
    out = q(torch.relu(z).float().cpu())                            # the saved post-ReLU activation, as stored
    mask = (out.double() > 0)
    if remask:      # the forward apply's own expression on the stored y: fma(y, a, b) > 0, a = rstd*gamma, b = beta - mean*a (fp32)
        a32 = rstd.float() * gamma.view(1, 1, C)
        b32 = beta.view(1, 1, C) - mean.float() * a32
        mask = (yd * a32.double() + b32.double()) > 0
        assert float((mask != (out.double() > 0)).double().mean()) <= (2e-3 if dt_name != 'F32' else 1e-5)   # the two masks differ only by storage underflow
    gsum = g0w[..., C:].double() + (g1.double() if two_grads else 0.0)
    dz = gsum * mask
    gd = gamma.double()
    s1 = (dz * gd).flatten(1).sum(1)
    s2 = (dz * gd * xhat).flatten(1).sum(1)
    dy_ref = rstd * (dz * gd - (s1 / cnt).view(N, 1, 1) - xhat * (s2 / cnt).view(N, 1, 1))
    dgamma_ref, dbeta_ref, dbias_ref = (dz * xhat).sum((0, 1)), dz.sum((0, 1)), dy_ref.sum((0, 1))

    sums = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    dgamma = torch.zeros(C, device='cuda'); dbeta = torch.zeros(C, device='cuda'); dbias = torch.zeros(C, device='cuda')
    dy = torch.zeros((N, nvox, 2 * C), dtype=tdt, device='cuda')     # written into the lower half of a 2C-wide buffer
    dres = torch.zeros((N, nvox, C), dtype=tdt, device='cuda')
    for p in range(2):
        L.call('seg3d_gn_bwd', dt, p, L.ptr(g0w, C), 2 * C, L.ptr(g1) if two_grads else None, C if two_grads else 0, None, 0,
               None if remask else L.ptr(out), C, L.ptr(y), C, C, L.ptr(stats), L.ptr(gamma), L.ptr(beta), eps, L.ptr(sums), L.ptr(dgamma), L.ptr(dbeta),
               L.ptr(dy), 2 * C, L.ptr(dres) if use_res else None, C if use_res else 0, L.ptr(dbias), N, nvox, L.stream_ptr())
    torch.cuda.synchronize()
    store = {'F32': 2e-6, 'BF16': 4.5e-3, 'F16': 6e-4}[dt_name]      # half an ulp of the stored type (2^-8, 2^-11) + fp32 arithmetic
    assert (dy[..., C:] == 0).all()
    err = (dy[..., :C].double() - dy_ref).abs().max() / dy_ref.abs().max()
    assert float(err) <= store + 1e-5, ('dy', float(err))
    if use_res:
        assert float((dres.double() - dz).abs().max() / dz.abs().max()) <= store, 'dres'
    for name, got, ref, mag in (('S1', sums[:, 0], s1, (dz * gd).abs().flatten(1).sum(1)), ('S2', sums[:, 1], s2, (dz * gd * xhat).abs().flatten(1).sum(1))):
        e = float(((got - ref).abs() / (mag + 1e-30)).max())
        assert e <= 2e-5, (name, e)
    for name, got, ref, mag in (('dgamma', dgamma, dgamma_ref, (dz * xhat).abs().sum((0, 1))), ('dbeta', dbeta, dbeta_ref, dz.abs().sum((0, 1))),
                                ('dbias', dbias, dbias_ref, dy_ref.abs().sum((0, 1)))):
        # fp32 accumulation of nvox*N terms per channel: compare against the sum of magnitudes; dbias sums the UNROUNDED dy
        e = float(((got.double() - ref).abs() / (mag + 1e-30)).max())
        assert e <= 2e-5, (name, e)
