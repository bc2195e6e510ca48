"""CPU check of the HOST WIRING of the standalone modules' training path (segmentation3d/_b200/blocks.py: run_module,
_ModuleFunction, _Tape) against the oracle's autograd.

The forward entry points are emulated as in tests/test_blocks_wiring.py, the backward ones as in
tests/test_autograd_wiring.py, and the two entry points the modules' backward adds are emulated here per
include/seg3d_b200.h: seg3d_gn_bwd_noact (the GroupNorm backward of a unit without ReLU) and the layout boundary
seg3d_grad_from_ncdhw / seg3d_grad_to_ncdhw (contributions summed in fp32, in argument order).  What runs for real is the
tape: which views feed which unit, the residual and skip windows, the dgrad convolutions on transformed weights, the
un-packing of the weight gradients.  Every parameter and input gradient of the eight module classes, and of VNet / VBNet
assembled from them, must equal the oracle's autograd gradient; the kernels themselves are pinned by
tests/test_gpu_blocks_train.py."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import net as onet
from test_autograd_wiring import _install as _install_backward
from test_blocks_wiring import _install as _install_blocks, _randomize
from test_plan_wiring import _mean_rstd, _rows

EPS = 1e-5
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
_BACKWARD = ('seg3d_gn_bwd', 'seg3d_conv3d_wgrad', 'seg3d_conv3d_cin1_wgrad', 'seg3d_outblock_tail_bwd')


def _install(monkeypatch):
    """forward emulations of the block tests + backward emulations of the whole-network tests + the two new entry points;
    returns the list of entry points called"""
    from segmentation3d._b200 import lib
    bw_calls = []
    _install_backward(monkeypatch, bw_calls)
    bw_call = lib.call
    _install_blocks(monkeypatch)
    fwd_call = lib.call
    calls = []

    def gn_bwd_noact(dtype, ps, g0, ld0, g1, ld1, g2, ld2, y, y_ld, C, stats, gamma, eps, sums, dgamma, dbeta,
                     dy, dy_ld, dres, dres_ld, dbias, N, nvox, stream):
        dz = _rows(g0, N * nvox, ld0, C).double()
        for g, ld in ((g1, ld1), (g2, ld2)):
            if g is not None:
                dz = dz + _rows(g, N * nvox, ld, C).double()
        dz = dz.view(N, nvox, C)
        mean, rstd = _mean_rstd(stats, float(nvox * C), eps, N)
        xh = (_rows(y, N * nvox, y_ld, C).double().view(N, nvox, C) - mean) * rstd
        gd = gamma.t.double().view(1, 1, C)
        st = sums.t.reshape(-1, 2)
        if ps == 0:
            st[:N, 0] += (dz * gd).flatten(1).sum(1)
            st[:N, 1] += (dz * gd * xh).flatten(1).sum(1)
            dgamma.t.reshape(-1)[dgamma.off:dgamma.off + C] += (dz * xh).sum((0, 1)).float()
            dbeta.t.reshape(-1)[dbeta.off:dbeta.off + C] += dz.sum((0, 1)).float()
        else:
            cnt = float(nvox * C)
            d = rstd * (gd * dz - (st[:N, 0] / cnt).view(N, 1, 1) - xh * (st[:N, 1] / cnt).view(N, 1, 1))
            dst = _rows(dy, N * nvox, dy_ld, C)
            dst.copy_(d.reshape(-1, C).to(dst.dtype))
            if dres is not None:
                r = _rows(dres, N * nvox, dres_ld, C)
                r.copy_(dz.reshape(-1, C).to(r.dtype))
            if dbias is not None:
                dbias.t.reshape(-1)[dbias.off:dbias.off + C] += d.sum((0, 1)).float()
        return 0

    def grad_to_ncdhw(dtype, n, g0, ld0, off0, g1, ld1, off1, g2, ld2, off2, C, N, nvox, out, stream):
        assert 1 <= n <= 3
        acc = torch.zeros((N * nvox, C), dtype=torch.float32)
        for g, ld, off in ((g0, ld0, off0), (g1, ld1, off1), (g2, ld2, off2))[:n]:
            assert ld >= off + C and g.t.dtype == lib.TORCH_DTYPE[dtype]
            acc += _rows(type(g)(g.t, g.off + off), N * nvox, ld, C).float()
        out.t.reshape(-1)[out.off:out.off + N * C * nvox].copy_(acc.view(N, nvox, C).permute(0, 2, 1).reshape(-1))
        return 0

    def grad_from_ncdhw(dtype, inp, C, N, nvox, out, ld, off, stream):
        assert ld >= off + C and out.t.dtype == lib.TORCH_DTYPE[dtype]
        src = inp.t.reshape(-1)[inp.off:inp.off + N * C * nvox].view(N, C, nvox).permute(0, 2, 1).reshape(-1, C)
        dst = _rows(type(out)(out.t, out.off + off), N * nvox, ld, C)
        dst.copy_(src.to(dst.dtype))
        return 0

    def wgrad_k1(mode, dtype, x, x_ld, Cin, dy, dy_ld, Cout, dw, N, D, H, W, stream):
        # the whole-network emulation covers k3 / k2s2 / t2s2; the 1x1x1 convolution's dw[ci][co] = sum_v x[v][ci] dy[v][co]
        n = N * D * H * W
        g = _rows(x, n, x_ld, Cin).double().t() @ _rows(dy, n, dy_ld, Cout).double()
        dw.t.reshape(-1)[dw.off:dw.off + Cin * Cout] += g.reshape(-1).float()
        return 0

    mine = {'seg3d_gn_bwd_noact': gn_bwd_noact, 'seg3d_grad_to_ncdhw': grad_to_ncdhw, 'seg3d_grad_from_ncdhw': grad_from_ncdhw}

    def call(name, *args):
        calls.append(name)
        if name in mine:
            assert mine[name](*args) == 0
        elif name == 'seg3d_conv3d_wgrad' and args[0] == lib.CONV_K1:
            assert wgrad_k1(*args) == 0
        elif name in _BACKWARD:
            bw_call(name, *args)
        else:
            fwd_call(name, *args)
    monkeypatch.setattr(lib, 'call', call)
    return calls


def _leaves(module, prefix):
    return {prefix + k: v.detach().clone().requires_grad_(True) for k, v in module.named_parameters()}


def _cases():
    """(name, module factory, input shapes, oracle(params, *inputs))"""
    from segmentation3d.network.module.conv_gn_relu3 import BottConvGnRelu3, ConvGnRelu3
    from segmentation3d.network.module.residual_block3 import BottResidualBlock3, ResidualBlock3
    from segmentation3d.network.module.vnet_downblock import DownBlock
    from segmentation3d.network.module.vnet_inblock import InputBlock
    from segmentation3d.network.module.vnet_outblock import OutputBlock
    from segmentation3d.network.module.vnet_upblock import UpBlock

    def cgr(stride, act, k=3, pad=1):
        def f(p, x):
            y = F.group_norm(F.conv3d(x, p['m.conv.weight'], p.get('m.conv.bias'), stride=stride, padding=pad), 1,
                             p['m.gn.weight'], p['m.gn.bias'], EPS)
            return F.relu(y) if act else y
        return f

    def tail(p, x):
        y = F.relu(F.group_norm(F.conv3d(x, p['m.conv1.weight'], p['m.conv1.bias'], padding=1), 1, p['m.gn1.weight'], p['m.gn1.bias'], EPS))
        return F.softmax(F.group_norm(F.conv3d(y, p['m.conv2.weight'], p['m.conv2.bias']), 1, p['m.gn2.weight'], p['m.gn2.bias'], EPS), 1)

    def bott(act):
        def f(p, x):
            y = onet._conv_gn(onet._conv_gn(x, p, 'm.conv1', True), p, 'm.conv2', True)
            return onet._conv_gn(y, p, 'm.conv3', act)
        return f

    return [
        ('ConvGnRelu3', lambda: ConvGnRelu3(16, 32, 3, 1, 1), [(2, 16, 4, 4, 8)], cgr(1, True)),
        ('ConvGnRelu3_noact', lambda: ConvGnRelu3(16, 32, 3, 1, 1, do_act=False), [(2, 16, 4, 4, 8)], cgr(1, False)),
        ('ConvGnRelu3_k2_nobias', lambda: ConvGnRelu3(16, 16, 2, 2, 0, bias=False), [(2, 16, 4, 4, 8)], cgr(2, True, 2, 0)),
        ('ConvGnRelu3_k1_noact', lambda: ConvGnRelu3(16, 16, 1, 1, 0, do_act=False), [(2, 16, 4, 4, 8)], cgr(1, False, 1, 0)),
        ('BottConvGnRelu3_noact', lambda: BottConvGnRelu3(32, 32, 3, 1, 1, 4, do_act=False), [(1, 32, 4, 4, 8)], bott(False)),
        ('BottConvGnRelu3', lambda: BottConvGnRelu3(32, 16, 3, 1, 1, 2), [(1, 32, 4, 4, 8)], bott(True)),
        ('ResidualBlock3', lambda: ResidualBlock3(32, 3, 1, 1, 2), [(2, 32, 4, 4, 8)], lambda p, x: onet._rblock(x, p, 'm')),
        ('ResidualBlock3_1', lambda: ResidualBlock3(16, 3, 1, 1, 1), [(2, 16, 4, 4, 8)], lambda p, x: onet._rblock(x, p, 'm')),
        ('BottResidualBlock3', lambda: BottResidualBlock3(64, 3, 1, 1, 4, 2), [(1, 64, 4, 4, 8)], lambda p, x: onet._rblock(x, p, 'm')),
        ('InputBlock', lambda: InputBlock(1, 16), [(2, 1, 8, 8, 8)], cgr(1, True)),
        ('DownBlock', lambda: DownBlock(32, 2), [(1, 32, 8, 8, 8)], lambda p, x: onet._down(x, p, 'm')),
        ('DownBlock_bott', lambda: DownBlock(32, 2, compression=True), [(1, 32, 8, 8, 8)], lambda p, x: onet._down(x, p, 'm')),
        ('UpBlock', lambda: UpBlock(128, 64, 2), [(1, 128, 2, 4, 4), (1, 32, 4, 8, 8)], lambda p, x, s: onet._up(x, s, p, 'm')),
        ('UpBlock_bott', lambda: UpBlock(64, 64, 1, compression=True), [(2, 64, 2, 2, 4), (2, 32, 4, 4, 8)],
         lambda p, x, s: onet._up(x, s, p, 'm')),
        ('OutputBlock', lambda: OutputBlock(32, 2), [(2, 32, 4, 4, 8)], tail),
        ('OutputBlock_5', lambda: OutputBlock(32, 5), [(1, 32, 4, 4, 8)], tail),
    ]


def _compare(got, ref, what, mode):
    assert got is not None and got.shape == ref.shape, what
    if mode == 'fp32':
        err = float((got - ref).abs().max()) / (float(ref.abs().max()) + 1e-12)
        assert err <= 1e-4, (what, err)
    else:       # bf16 storage of activations and gradients: direction (on a few hundred voxels; the GPU test uses more)
        a, b = ref.double().flatten(), got.double().flatten()
        cos = float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-30))
        assert cos >= 0.98, (what, cos)


@pytest.mark.parametrize('mode', ['fp32', 'bf16'])
def test_every_module_class_differentiates_like_oracle_autograd(monkeypatch, mode):
    calls = _install(monkeypatch)
    monkeypatch.setenv('SEG3D_MODE', mode)
    g = torch.Generator().manual_seed(3)
    for name, make, shapes, oracle in _cases():
        m = make()
        _randomize(m, 11)
        xs = [torch.randn(s, generator=g) for s in shapes]
        params = _leaves(m, 'm.')
        xr = [x.clone().requires_grad_(True) for x in xs]
        ref = oracle(params, *xr)
        r = torch.randn(ref.shape, generator=g)
        (ref * r).sum().backward()
        xg = [x.clone().requires_grad_(True) for x in xs]
        del calls[:]
        out = m(*xg)
        assert out.grad_fn is not None and out.dtype == torch.float32, name
        (out * r).sum().backward()
        for k, p in m.named_parameters():
            _compare(p.grad, params['m.' + k].grad, (name, k), mode)
        for i, (a, b) in enumerate(zip(xg, xr)):
            _compare(a.grad, b.grad, (name, 'input %d' % i), mode)
        assert ('seg3d_gn_bwd_noact' in calls) == name.endswith('_noact'), name
        assert calls.count('seg3d_grad_to_ncdhw') == len(xs), name
        assert calls.count('seg3d_grad_from_ncdhw') == (0 if name.startswith('OutputBlock') else 1), name


def test_input_gradient_only_when_asked(monkeypatch):
    """ctx.needs_input_grad: no data gradient of the first unit and no boundary launch for an input without grad; the
    parameter gradients do not change"""
    from segmentation3d.network.module.vnet_upblock import UpBlock
    calls = _install(monkeypatch)
    monkeypatch.setenv('SEG3D_MODE', 'fp32')
    m = UpBlock(64, 64, 1)
    _randomize(m, 5)
    g = torch.Generator().manual_seed(4)
    x, s = torch.randn((1, 64, 2, 2, 4), generator=g), torch.randn((1, 32, 4, 4, 8), generator=g)
    r = torch.randn((1, 64, 4, 4, 8), generator=g)
    grads = []
    for need in ((True, True), (False, True), (False, False)):
        m.zero_grad()
        del calls[:]
        xa, sa = x.clone().requires_grad_(need[0]), s.clone().requires_grad_(need[1])
        (m(xa, sa) * r).sum().backward()
        assert (xa.grad is not None) == need[0] and (sa.grad is not None) == need[1]
        assert calls.count('seg3d_grad_to_ncdhw') == sum(need)
        # dgrad convolutions: the residual unit's always (it feeds the up unit), the up unit's only for the input
        assert calls.count('seg3d_conv3d_fwd') == 2 + 1 + need[0]
        grads.append([p.grad.clone() for p in m.parameters()])
    for a, b in zip(grads[0], grads[2]):
        assert torch.equal(a, b)


def _vnet_forward(net, x):
    """reference network/vnet.py:36-48 over the drop-in blocks"""
    o16 = net.in_block(x)
    o32 = net.down_32(o16)
    o64 = net.down_64(o32)
    o128 = net.down_128(o64)
    o256 = net.down_256(o128)
    o = net.up_256(o256, o128)
    o = net.up_128(o, o64)
    o = net.up_64(o, o32)
    o = net.up_32(o, o16)
    return net.out_block(o)


@pytest.mark.parametrize('compression,cout', [(False, 2), (True, 3)])
def test_block_built_vnet_differentiates_like_the_oracle_net(monkeypatch, compression, cout):
    from test_abi_and_host import _assemble_from_blocks
    _install(monkeypatch)
    monkeypatch.setenv('SEG3D_MODE', 'fp32')
    torch.manual_seed(0)
    net = _assemble_from_blocks(1, cout, compression)
    # a pre-activation within ~1e-7 of 0 flips its ReLU between two fp32 evaluation orders and moves whole gradient tensors
    # by ~1e-2 (seed 8 has one); this seed has no such near-tie, so the two programs agree to fp32 rounding
    _randomize(net, 11)
    g = torch.Generator().manual_seed(12)
    x = torch.randn((1, 1, 16, 16, 16), generator=g)
    params = {k: v.detach().clone().requires_grad_(True) for k, v in net.named_parameters()}
    ref = onet.forward_with_grad(params, x)
    r = torch.randn(ref.shape, generator=g)
    (ref * r).sum().backward()
    out = _vnet_forward(net, x)
    assert float((out - ref).abs().max()) <= 1e-5
    (out * r).sum().backward()
    for k, p in net.named_parameters():
        _compare(p.grad, params[k].grad, k, 'fp32')


def test_training_refuses_more_than_16_classes_and_no_grad_launches_are_unchanged(monkeypatch):
    """OutputBlock(32, 20) refuses a training forward with the whole network's message; under torch.no_grad() every module
    issues exactly the launches (entry points and scalar arguments) it issued before it could train"""
    from segmentation3d.network.module.vnet_outblock import OutputBlock
    _install(monkeypatch)
    monkeypatch.setenv('SEG3D_MODE', 'bf16')
    with pytest.raises(RuntimeError, match='training supports up to 16 classes'):
        OutputBlock(32, 20)(torch.zeros((1, 32, 4, 4, 8)))
    monkeypatch.undo()
    got = _record_no_grad_launches(monkeypatch)
    with open(os.path.join(GOLDEN, 'blocks_nograd_launches.json')) as f:
        want = json.load(f)
    assert sorted(got) == sorted(want)
    for k in want:
        assert got[k] == want[k], k


def _record_no_grad_launches(monkeypatch):
    from segmentation3d._b200 import lib
    from segmentation3d.network.module.conv_gn_relu3 import BottConvGnRelu3, ConvGnRelu3
    from segmentation3d.network.module.residual_block3 import BottResidualBlock3, ResidualBlock3
    from segmentation3d.network.module.vnet_downblock import DownBlock
    from segmentation3d.network.module.vnet_inblock import InputBlock
    from segmentation3d.network.module.vnet_outblock import OutputBlock
    from segmentation3d.network.module.vnet_upblock import UpBlock
    _install_blocks(monkeypatch)
    inner = lib.call
    log = []

    def call(name, *args):
        log.append([name] + [a if isinstance(a, (int, float)) else (None if a is None else 'p') for a in args])
        return inner(name, *args)
    monkeypatch.setattr(lib, 'call', call)
    out = {}
    for mode in ('fp32', 'fp16', 'bf16'):
        monkeypatch.setenv('SEG3D_MODE', mode)
        g = torch.Generator().manual_seed(0)

        def r(*s):
            return torch.randn(s, generator=g)
        for name, m, xs in (('ConvGnRelu3', ConvGnRelu3(16, 32, 3, 1, 1, do_act=False), (r(2, 16, 4, 4, 8),)),
                            ('ConvGnRelu3_k2', ConvGnRelu3(16, 16, 2, 2, 0), (r(2, 16, 4, 4, 8),)),
                            ('ConvGnRelu3_k1', ConvGnRelu3(16, 16, 1, 1, 0, bias=False), (r(2, 16, 4, 4, 8),)),
                            ('BottConvGnRelu3', BottConvGnRelu3(32, 32, 3, 1, 1, 4, do_act=False), (r(1, 32, 4, 4, 8),)),
                            ('ResidualBlock3', ResidualBlock3(32, 3, 1, 1, 2), (r(2, 32, 4, 4, 8),)),
                            ('BottResidualBlock3', BottResidualBlock3(64, 3, 1, 1, 4, 2), (r(1, 64, 4, 4, 8),)),
                            ('InputBlock', InputBlock(1, 16), (r(2, 1, 8, 8, 8),)),
                            ('DownBlock', DownBlock(32, 2, compression=True), (r(1, 32, 8, 8, 8),)),
                            ('UpBlock', UpBlock(128, 64, 2), (r(1, 128, 2, 4, 4), r(1, 32, 4, 8, 8))),
                            ('OutputBlock', OutputBlock(32, 5), (r(2, 32, 4, 4, 8),))):
            _randomize(m, 1)
            del log[:]
            with torch.no_grad():
                m(*xs)
            out['%s/%s' % (mode, name)] = list(log)
    return out
