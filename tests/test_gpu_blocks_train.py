"""GPU checks of the standalone modules' training path (segmentation3d/_b200/blocks.py) on one B200:

  * seg3d_gn_bwd_noact against the float64 closed form (the bars seg3d_gn_bwd meets in tests/test_gpu_kernels.py);
  * seg3d_grad_to_ncdhw / seg3d_grad_from_ncdhw bit-exact against the fp32 sum in the kernel's order, memory outside the
    written window untouched;
  * every parameter and input gradient of each module class (fp32, on inputs without a ReLU near-tie: worst error <= 1e-4
    of each tensor's max; bf16: cosine >= 0.995, 0.98 for bottleneck stacks) and of a block-built VNet at 2 x 32^3 (fp32:
    parameters within 1e-2, the input gradient's direction) against float64 autograd of the oracle;
  * three seg_train.train_step's with FlatAdam on a block-built VNet; OutputBlock(32, 20) refuses training.
The host wiring alone is pinned on the CPU by tests/test_blocks_train_wiring.py."""
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import net as onet
from test_blocks_train_wiring import _cases, _vnet_forward
from test_blocks_wiring import _randomize

pytestmark = [pytest.mark.gpu]


@pytest.fixture(scope='module')
def lib():
    from segmentation3d._b200 import lib as L
    assert L.load().seg3d_device_check(0) == 0, L.load().seg3d_last_error()
    return L


@pytest.mark.parametrize('dt_name', ['F32', 'BF16', 'F16'])
@pytest.mark.parametrize('C,nvox,n_grads', [(16, 517, 1), (32, 1000, 3), (64, 96, 2), (256, 40, 1)])
def test_gn_bwd_noact_matches_closed_form(lib, dt_name, C, nvox, n_grads):
    """seg3d_gn_bwd_noact (both passes): dz = g0 + g1 + g2 unmasked, against float64 on the same stored tensors: dy and dres
    within half an ulp of the stored type, the per-sample sums, dgamma, dbeta and dbias within 2e-5 of the sum of the
    magnitudes of their terms.  Contribution 0 lives in the upper half of a 2C-wide buffer, dy is written into the lower
    half of one."""
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N, eps = 2, 1e-5
    g = torch.Generator().manual_seed(7 * C + nvox)
    q = lambda t: t.to(tdt).cuda()                                  # noqa: E731  (stored tensors)
    y = q(torch.randn((N, nvox, C), generator=g) * 1.5 + 0.3)
    gamma = torch.randn(C, generator=g).cuda() + 1.0
    g0w = q(torch.randn((N, nvox, 2 * C), generator=g) * 1e-3)
    gs = [q(torch.randn((N, nvox, C), generator=g) * 1e-3) for _ in range(2)]
    yd = y.double()
    cnt = float(nvox * C)
    stats = torch.stack([yd.flatten(1).sum(1), (yd * yd).flatten(1).sum(1)], 1).contiguous()
    mean = (stats[:, 0] / cnt).view(N, 1, 1)
    rstd = 1.0 / torch.sqrt((stats[:, 1] / cnt).view(N, 1, 1) - mean * mean + eps)
    xhat = (yd - mean) * rstd
    dz = g0w[..., C:].double()
    for k in range(n_grads - 1):
        dz = dz + gs[k].double()
    gd = gamma.double()
    s1, s2 = (dz * gd).flatten(1).sum(1), (dz * gd * xhat).flatten(1).sum(1)
    dy_ref = rstd * (dz * gd - (s1 / cnt).view(N, 1, 1) - xhat * (s2 / cnt).view(N, 1, 1))

    sums = torch.zeros((N, 2), dtype=torch.float64, device='cuda')
    dgamma, dbeta, dbias = (torch.zeros(C, device='cuda') for _ in range(3))
    dy = torch.zeros((N, nvox, 2 * C), dtype=tdt, device='cuda')
    dres = torch.zeros((N, nvox, C), dtype=tdt, device='cuda')
    g1 = gs[0] if n_grads > 1 else None
    g2 = gs[1] if n_grads > 2 else None
    for p in range(2):
        L.call('seg3d_gn_bwd_noact', dt, p, L.ptr(g0w, C), 2 * C, L.ptr(g1), C if g1 is not None else 0, L.ptr(g2),
               C if g2 is not None else 0, L.ptr(y), C, C, L.ptr(stats), L.ptr(gamma), eps, L.ptr(sums), L.ptr(dgamma),
               L.ptr(dbeta), L.ptr(dy), 2 * C, L.ptr(dres), C, L.ptr(dbias), N, nvox, L.stream_ptr())
    torch.cuda.synchronize()
    store = {'F32': 2e-6, 'BF16': 4.5e-3, 'F16': 6e-4}[dt_name]      # half an ulp of the stored type (2^-8, 2^-11) + fp32 arithmetic
    assert (dy[..., C:] == 0).all()
    err = float((dy[..., :C].double() - dy_ref).abs().max() / dy_ref.abs().max())
    assert err <= store + 1e-5, ('dy', err)
    assert float((dres.double() - dz).abs().max() / dz.abs().max()) <= store, 'dres'
    for name, got, ref, mag in (('S1', sums[:, 0], s1, (dz * gd).abs().flatten(1).sum(1)),
                                ('S2', sums[:, 1], s2, (dz * gd * xhat).abs().flatten(1).sum(1)),
                                ('dgamma', dgamma.double(), (dz * xhat).sum((0, 1)), (dz * xhat).abs().sum((0, 1))),
                                ('dbeta', dbeta.double(), dz.sum((0, 1)), dz.abs().sum((0, 1))),
                                ('dbias', dbias.double(), dy_ref.sum((0, 1)), dy_ref.abs().sum((0, 1)))):
        e = float(((got - ref).abs() / (mag + 1e-30)).max())
        assert e <= 2e-5, (name, e)


@pytest.mark.parametrize('dt_name', ['F32', 'BF16', 'F16'])
@pytest.mark.parametrize('C,nvox,layout', [
    (32, 1000, [(48, 16), (32, 0), (64, 8)]),       # padded pitches, nonzero channel offsets, three contributions
    (64, 333, [(128, 64), (64, 0)]),                 # ragged nvox, the skip half of a concat gradient
    (16, 4096, [(16, 0)]),
    (256, 130, [(256, 0), (512, 256), (256, 0)]),
    (1, 517, [(1, 0)]),                              # the input block's one-channel data gradient: scalar path
    (24, 301, [(27, 3), (24, 0)]),                   # pitch / offset not a whole 16-byte vector: scalar path
])
def test_grad_boundary_is_bit_exact_and_stays_in_its_window(lib, dt_name, C, nvox, layout):
    L = lib
    dt = getattr(L, dt_name)
    tdt = L.TORCH_DTYPE[dt]
    N = 2
    g = torch.Generator().manual_seed(C + nvox)
    bufs = [torch.randn((N, nvox, ld), generator=g).to(tdt).cuda() for ld, _ in layout]
    ref = torch.zeros((N * nvox, C), dtype=torch.float32)
    for b, (ld, off) in zip(bufs, layout):          # the kernel's order: ((0 + g0) + g1) + g2 in fp32
        ref = ref + b.cpu().float().reshape(-1, ld)[:, off:off + C]
    ref = ref.view(N, nvox, C).permute(0, 2, 1).contiguous()
    guard = 777
    out = torch.full((N * C * nvox + guard,), float('nan'), device='cuda')
    args = []
    for k in range(3):
        if k < len(layout):
            args += [L.ptr(bufs[k]), layout[k][0], layout[k][1]]
        else:
            args += [None, 0, 0]
    L.call('seg3d_grad_to_ncdhw', dt, len(layout), *args, C, N, nvox, L.ptr(out), L.stream_ptr())
    torch.cuda.synchronize()
    got = out[:N * C * nvox].view(N, C, nvox).cpu()
    assert torch.equal(got, ref)
    assert torch.isnan(out[N * C * nvox:]).all()

    # NCDHW fp32 -> a channel window of an NDHWC buffer in the storage type
    ld, off = layout[-1]
    src = torch.randn((N, C, nvox), generator=g).cuda()
    dst = torch.full((N, nvox, ld + 8 if off + C == ld else ld), float('nan'), device='cuda').to(tdt)
    L.call('seg3d_grad_from_ncdhw', dt, L.ptr(src), C, N, nvox, L.ptr(dst), dst.shape[-1], off, L.stream_ptr())
    torch.cuda.synchronize()
    d = dst.cpu()
    assert torch.equal(d[..., off:off + C], src.cpu().permute(0, 2, 1).to(tdt))
    assert torch.isnan(d[..., :off].float()).all() and torch.isnan(d[..., off + C:].float()).all()


def _f64_grads(m, oracle, xs, r):
    """float64 autograd of the oracle's restatement of module m: (parameter grads by name, input grads)"""
    params = {'m.' + k: v.detach().cpu().double().requires_grad_(True) for k, v in m.named_parameters()}
    xd = [x.detach().cpu().double().requires_grad_(True) for x in xs]
    (oracle(params, *xd) * r.double()).sum().backward()
    return {k[2:]: v.grad for k, v in params.items()}, [x.grad for x in xd]


def _check(got, ref, what, mode, bar):
    """fp32: worst error over the tensor's max <= bar; bf16: cosine >= bar.  Returns a failure message or None."""
    got = got.detach().cpu().double()
    assert got.shape == ref.shape, what
    if mode == 'fp32':
        err = float((got - ref).abs().max()) / (float(ref.abs().max()) + 1e-30)
        print(what, 'rel err %.2e' % err)
        return None if err <= bar else '%s rel err %.3g > %g' % (what, err, bar)
    a, b = ref.flatten(), got.flatten()
    cos = float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-300))
    print(what, 'cosine %.5f' % cos)
    return None if cos >= bar else '%s cosine %.5f < %g' % (what, cos, bar)


def _tie_margin(oracle, m, xs):
    """smallest |ReLU input| of the float64 oracle over that input's max |value|: below ~1e-6 the fp32 kernels and the
    float64 program may put that voxel on different sides of the ReLU, which moves whole gradient tensors by ~1e-3..1e-2"""
    params = {'m.' + k: v.detach().cpu().double() for k, v in m.named_parameters()}
    worst, real = [float('inf')], F.relu

    def relu(t, inplace=False):
        worst[0] = min(worst[0], float(t.abs().min() / t.abs().max()))
        return real(t)
    F.relu = relu
    try:
        with torch.no_grad():
            oracle(params, *[x.double() for x in xs])
    finally:
        F.relu = real
    return worst[0]


# bf16: DESIGN.md section 2 gives cosine >= 0.995 for well-conditioned layers; a bottleneck stack (BottConvGnRelu3, and
# the residual / down / up blocks built from it) chains three to six GroupNorm -> ReLU units on 8-16 channels, where bf16
# rounding of the stored activations flips ReLU masks (the band of the whole network's deep layers, cosine 0.966-0.99):
# the CPU emulation with bf16 storage and exact arithmetic already lands at cosine 0.99 there, so those are held to 0.98
_BF16_BAR = {'BottConvGnRelu3': 0.98, 'BottConvGnRelu3_noact': 0.98, 'BottResidualBlock3': 0.98, 'DownBlock_bott': 0.98,
             'UpBlock_bott': 0.98}


@pytest.mark.parametrize('mode', ['fp32', 'bf16'])
def test_every_module_class_gradient_against_float64(monkeypatch, mode):
    monkeypatch.setenv('SEG3D_MODE', mode)
    failures = []
    for name, make, shapes, oracle in _cases():
        m = make()
        _randomize(m, 11)
        if mode == 'bf16':      # twice the wiring test's extent per spatial dim: more voxels per GroupNorm and weight gradient
            shapes = [s[:2] + tuple(2 * d for d in s[2:]) for s in shapes]
        for seed in range(40):  # fp32: inputs without a ReLU near-tie (see _tie_margin)
            g = torch.Generator().manual_seed(seed)
            xs = [torch.randn(s, generator=g) for s in shapes]
            if mode == 'bf16' or _tie_margin(oracle, m, xs) >= 3e-6:
                break
        else:
            pytest.fail('%s: no tie-free input in 40 draws' % name)
        m = m.cuda()
        xg = [x.cuda().requires_grad_(True) for x in xs]
        out = m(*xg)
        r = torch.randn(out.shape, generator=g)
        (out * r.cuda()).sum().backward()
        pref, xref = _f64_grads(m, oracle, xs, r)
        bar = 1e-4 if mode == 'fp32' else _BF16_BAR.get(name, 0.995)
        for k, p in m.named_parameters():
            failures.append(_check(p.grad, pref[k], (name, k), mode, bar))
        for i, x in enumerate(xg):
            failures.append(_check(x.grad, xref[i], (name, 'input %d' % i), mode, bar))
    failures = [f for f in failures if f]
    assert not failures, failures


def _block_vnet(compression, cout, seed):
    from test_abi_and_host import _assemble_from_blocks
    torch.manual_seed(seed)
    net = _assemble_from_blocks(1, cout, compression)
    net.forward = types.MethodType(_vnet_forward, net)
    return net


def test_block_built_vnet_gradient_against_float64(monkeypatch):
    monkeypatch.setenv('SEG3D_MODE', 'fp32')
    net = _block_vnet(False, 2, 0)
    _randomize(net, 11)
    g = torch.Generator().manual_seed(12)
    x = torch.randn((2, 1, 32, 32, 32), generator=g)
    params = {k: v.detach().double().requires_grad_(True) for k, v in net.named_parameters()}
    xd = x.double().requires_grad_(True)
    ref = onet.forward_with_grad(params, xd)
    r = torch.randn(ref.shape, generator=g)
    (ref * r.double()).sum().backward()
    net = net.cuda()
    xg = x.cuda().requires_grad_(True)
    out = net(xg)
    assert float((out.detach().cpu().double() - ref.detach()).abs().max()) <= 1e-4
    (out * r.cuda()).sum().backward()
    # 2 x 32^3 carries ~10^7 ReLU inputs: some lie within fp32 rounding of 0 and flip against float64 (see _tie_margin), moving
    # the gradients below them by up to ~1e-2 of their max, the bar the whole network's fp32 gradient test uses too
    # (tests/test_gpu_train.py); tie-free inputs hold 1e-4 in the module test above and in tests/test_blocks_train_wiring.py
    failures = [_check(p.grad, params[k].grad, k, 'fp32', 1e-2) for k, p in net.named_parameters()]
    failures.append(_check(xg.grad, xd.grad, 'input', 'bf16', 0.999))     # every flip lands here: its direction
    failures = [f for f in failures if f]
    assert not failures, failures


def test_three_train_steps_with_flat_adam_on_a_block_built_vnet(monkeypatch):
    from segmentation3d.core.seg_train import make_optimizer, train_step
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    monkeypatch.setenv('SEG3D_MODE', 'bf16')
    net = _block_vnet(False, 2, 0).cuda()
    net.train()
    opt = make_optimizer(net, 1e-3)
    g = torch.Generator().manual_seed(3)
    crops = torch.randn((2, 1, 32, 32, 32), generator=g).cuda()
    masks = (torch.rand((2, 1, 32, 32, 32), generator=g) > 0.7).float().cuda()
    before = [p.detach().clone() for p in net.parameters()]
    lf = MultiDiceLoss([1.0, 1.0], 2, True)
    losses = [float(train_step(net, opt, lf, crops, masks)) for _ in range(3)]
    print('losses', losses)
    assert losses[2] < losses[0], losses
    for (k, p), b in zip(net.named_parameters(), before):
        assert not torch.equal(p.detach(), b), k


def test_output_block_above_16_classes_infers_but_refuses_training(monkeypatch):
    from segmentation3d.network.module.vnet_outblock import OutputBlock
    monkeypatch.setenv('SEG3D_MODE', 'bf16')
    m = OutputBlock(32, 20).cuda()
    x = torch.randn((1, 32, 8, 8, 16), device='cuda')
    with pytest.raises(RuntimeError, match='training supports up to 16 classes'):
        m(x)
    with torch.no_grad():
        p = m(x)
    assert p.shape == (1, 20, 8, 8, 16) and float((p.sum(1) - 1).abs().max()) <= 1e-4
