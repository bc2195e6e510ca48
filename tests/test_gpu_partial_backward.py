"""B200 checks of the whole network's partial backward: seg3d_conv3d_cin1_dgrad against float64, the input gradient of VNet and
VBNet, and frozen-encoder fine-tuning through seg_train.make_optimizer / train_step."""
import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from oracle import net as onet

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -23
TERMS = 27 * 16 + 2          # 27 x 16 fp32 products per output voxel, plus two roundings of slack


def _lib():
    from segmentation3d._b200 import lib
    lib.load()
    return lib


def _ref_dgrad(gy, w):
    """float64 dx and sum |w||gy| per voxel.  gy: [N,D,H,W,16]; w: [27][16] fp32 (tap-major)"""
    g = gy.double().permute(0, 4, 1, 2, 3)
    wk = w.double().view(3, 3, 3, 16).permute(3, 0, 1, 2).unsqueeze(1)
    return F.conv_transpose3d(g, wk, padding=1)[:, 0], F.conv_transpose3d(g.abs(), wk.abs(), padding=1)[:, 0]


@pytest.mark.parametrize('shape', [(1, 16, 16, 16), (2, 16, 32, 48), (3, 16, 16, 16), (2, 96, 96, 96)])
@pytest.mark.parametrize('dtype', ['f16', 'bf16', 'f32'])
@pytest.mark.parametrize('ld', [16, 32])
def test_cin1_dgrad_against_float64(shape, dtype, ld):
    L = _lib()
    dt, td = {'f16': (L.F16, torch.float16), 'bf16': (L.BF16, torch.bfloat16), 'f32': (L.F32, torch.float32)}[dtype]
    N, D, H, W = shape
    g = torch.Generator(device='cuda').manual_seed(N * 1000 + D + ld)
    buf = torch.full((N, D, H, W, ld), float('nan'), device='cuda', dtype=td)
    buf[..., :16] = torch.randn((N, D, H, W, 16), generator=g, device='cuda').to(td)       # channels >= 16 stay NaN: unread
    w = (torch.randn((27, 16), generator=g, device='cuda') * 0.2).contiguous()
    pad = 64
    out = torch.full((N * D * H * W + 2 * pad,), float('nan'), device='cuda')
    L.call('seg3d_conv3d_cin1_dgrad', dt, L.ptr(buf), ld, L.ptr(w), L.ptr(out, pad), N, D, H, W, L.stream_ptr())
    torch.cuda.synchronize()
    assert torch.isnan(out[:pad]).all() and torch.isnan(out[-pad:]).all(), 'wrote outside [N,1,D,H,W]'
    ref, mag = _ref_dgrad(buf[..., :16].float(), w)
    got = out[pad:-pad].view(N, D, H, W).double()
    excess = float(((got - ref).abs() - EPS32 * TERMS * mag).max())
    assert excess <= 0, excess


def _sd(arch, cout, seed=0):
    return oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, seed), 5)


def _net(arch, cout, mode, sd):
    import importlib
    net = importlib.import_module('segmentation3d.network.' + arch).SegmentationNet(1, cout)
    net.load_state_dict(sd)
    net.b200_mode = mode
    return net.cuda().train()


def _input_grad(net, x, r, freeze=True):
    for p in net.parameters():
        p.requires_grad_(not freeze)
    xg = x.clone().requires_grad_(True)
    (net(xg) * r).sum().backward()
    return xg.grad


def _in_block_stage(net, xgrad):
    """excess of the returned input gradient over the seg3d_conv3d_cin1_dgrad bound, recomputed in float64 from the gy
    buffer the kernel read"""
    plan = net._plan
    B, _, D, H, W = xgrad.shape
    bw = plan._plans[(B, D, H, W, True)][0]['bwd']
    gy = bw.gy['in_block.conv']
    ref, mag = _ref_dgrad(gy.buf.view(B, D, H, W, gy.ld)[..., :16].float(), plan.convs['in_block.conv'].w.view(27, 16))
    return float(((xgrad[:, 0].double() - ref).abs() - EPS32 * TERMS * mag).max())


@pytest.mark.parametrize('arch,cout', [('vnet', 2), ('vbnet', 3)])
def test_input_gradient_of_the_network(arch, cout):
    _lib()
    sd = _sd(arch, cout)
    g = torch.Generator().manual_seed(3)
    x = torch.randn((2, 1, 32, 32, 32), generator=g)
    r = torch.randn((2, cout, 32, 32, 32), generator=g)
    # float64 autograd of the oracle
    params = {k: v.double() for k, v in sd.items()}
    xd = x.double().requires_grad_(True)
    (onet.forward_with_grad(params, xd) * r.double()).sum().backward()
    ref = xd.grad
    n32 = _net(arch, cout, 'fp32', sd)
    g32 = _input_grad(n32, x.cuda(), r.cuda())
    assert _in_block_stage(n32, g32) <= 0            # seg3d_conv3d_cin1_dgrad on fp32 gy, to its bound
    g32 = g32.cpu().double()
    # 2 x 32^3 carries ~10^7 ReLU inputs, some within fp32 rounding of 0 that flip against float64 (tests/test_gpu_blocks_train.py
    # explains the band): the whole-network bar is that of the block-built VNet there, 1e-2 of the max and cosine 0.999
    err = float((g32 - ref).abs().max()) / float(ref.abs().max())
    cos = float(torch.dot(g32.flatten(), ref.flatten()) / (g32.norm() * ref.norm()))
    print(arch, 'fp32 input gradient: rel err %.2e, cosine %.6f' % (err, cos))
    assert err <= 1e-2 and cos >= 0.999, (err, cos)
    # bf16: the in-block stage to its bound, the whole chain by direction against the fp32 mode.  The input gradient crosses
    # every layer, and bf16 storage alone puts the deep layers' gradients at cosine 0.966-0.99 (DESIGN.md section 2); VNet's
    # input gradient measured 0.989 on B200, so the chain is held to 0.98, the bar of the bottleneck stacks in
    # tests/test_gpu_blocks_train.py
    nb = _net(arch, cout, 'bf16', sd)
    gb = _input_grad(nb, x.cuda(), r.cuda())
    assert _in_block_stage(nb, gb) <= 0
    gb = gb.cpu().double()
    cos = float(torch.dot(gb.flatten(), g32.flatten()) / (gb.norm() * g32.norm()))
    print(arch, 'bf16 input gradient cosine vs fp32 mode %.5f' % cos)
    assert cos >= 0.98, cos
    # every parameter trainable as well: the same input gradient, and the parameters still get theirs
    nb2 = _net(arch, cout, 'bf16', sd)
    gb2 = _input_grad(nb2, x.cuda(), r.cuda(), freeze=False)
    assert all(p.grad is not None for p in nb2.parameters())
    assert _in_block_stage(nb2, gb2) <= 0


def test_input_gradient_at_the_benchmark_shape():
    _lib()
    sd = _sd('vnet', 2)
    net = _net('vnet', 2, 'bf16', sd)
    g = torch.Generator(device='cuda').manual_seed(4)
    x = torch.randn((8, 1, 96, 96, 96), generator=g, device='cuda')
    r = torch.randn((8, 2, 96, 96, 96), generator=g, device='cuda')
    gx = _input_grad(net, x, r)
    assert torch.isfinite(gx).all()
    assert _in_block_stage(net, gx) <= 0


def test_frozen_encoder_fine_tuning():
    from segmentation3d.core.seg_train import make_optimizer, train_step
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    _lib()
    sd = _sd('vnet', 2)
    g = torch.Generator().manual_seed(6)
    crops = torch.randn((2, 1, 32, 32, 32), generator=g).cuda()
    masks = (crops > 0.3).float()
    lf = MultiDiceLoss([1.0, 1.0], 2, False)
    enc = ('in_block', 'down_')
    # the all-trainable backward of the same forward
    full = _net('vnet', 2, 'bf16', sd)
    lf(full(crops), masks).backward()
    ref = {n: p.grad.clone() for n, p in full.named_parameters()}
    net = _net('vnet', 2, 'bf16', sd)
    for n, p in net.named_parameters():
        p.requires_grad_(not n.startswith(enc))
    opt = make_optimizer(net, 1e-3)
    before = {n: p.detach().clone() for n, p in net.named_parameters()}
    losses = []
    for step in range(3):
        losses.append(float(train_step(net, opt, lf, crops, masks)))
        if step == 0:
            for n, p in net.named_parameters():
                if n.startswith(enc):
                    assert p.grad is None, n
                else:       # the fp32 weight-gradient bound of tests/test_gpu_train_stages.py, relative to the tensor's max
                    err = float((p.grad - ref[n]).abs().max()) / (float(ref[n].abs().max()) + 1e-30)
                    assert err <= 2e-5, (n, err)
    torch.cuda.synchronize()
    for n, p in net.named_parameters():
        if n.startswith(enc):
            assert torch.equal(p.detach(), before[n]), n
        else:
            assert not torch.equal(p.detach(), before[n]), n
    print('losses', losses)
    assert losses[-1] < losses[0], losses


def test_ranged_adam_against_torch_adam():
    """seg3d_adam_step_ranges through FlatAdam: 80 parameters (odd sizes), a freeze pattern that changes every step so the
    step counts differ between neighbours and one step issues more than 32 ranges (two launches), weight decay on; every
    parameter and both moments against torch.optim.Adam on the same gradients, frozen entries bit-identical.
    The betas are exact in fp32 (0.875, 1 - 2^-10): the kernels take them as fp32 and form 1 - beta there, which for
    beta2 = 0.999 differs from torch's double 1 - beta2 by 1.3e-5 relative - a property of seg3d_adam_step's arithmetic
    that the ranged entry shares, so that a parameter's update does not depend on which entry ran it."""
    from segmentation3d._b200.optim import FlatAdam
    _lib()
    g = torch.Generator().manual_seed(7)
    shapes = [((i % 7) * 5 + 1, (i % 3) + 1) for i in range(80)]
    init = [torch.randn(s, generator=g) for s in shapes]
    ours = [t.clone().cuda().requires_grad_(True) for t in init]
    ref = [t.clone().cuda().requires_grad_(True) for t in init]
    betas = (0.875, 1.0 - 2.0 ** -10)
    opt = FlatAdam(ours, lr=1e-2, betas=betas, weight_decay=1e-2)
    topt = torch.optim.Adam(ref, lr=1e-2, betas=betas, weight_decay=1e-2, foreach=False)
    most = 0
    for step in range(6):
        frozen = {i for i in range(80) if (i + step) % 3 == 0 or (step == 0 and i < 40)}
        held = {i: (ours[i].detach().clone(), ours[i] in opt.state and opt.state[ours[i]].get('exp_avg') is not None and
                    opt.state[ours[i]]['exp_avg'].clone()) for i in frozen}
        for i, (a, b) in enumerate(zip(ours, ref)):
            gr = torch.randn(shapes[i], generator=g).cuda()
            a.grad = None if i in frozen else gr.clone()
            b.grad = None if i in frozen else gr.clone()
        opt.step()
        topt.step()
        torch.cuda.synchronize()
        most = max(most, len(opt._ranges([i not in frozen for i in range(80)])))      # the table this step used
        for i, (a, b) in enumerate(zip(ours, ref)):
            if i in frozen:
                assert torch.equal(a.detach(), held[i][0]), (step, i)
                if held[i][1] is not False:
                    assert torch.equal(opt.state[a]['exp_avg'], held[i][1]), (step, i)
            err = float((a.detach() - b.detach()).abs().max())
            assert err <= 1e-6 * float(b.detach().abs().max()), (step, i, err)
            if b in topt.state:
                assert float(opt.state[a]['step']) == float(topt.state[b]['step']), (step, i)
                for k in ('exp_avg', 'exp_avg_sq'):
                    rm = topt.state[b][k]
                    assert float((opt.state[a][k] - rm).abs().max()) <= 1e-6 * float(rm.abs().max()) + 1e-30, (step, i, k)
    assert most > 32, most                       # some step needed two launches
