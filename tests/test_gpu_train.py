"""GPU parity of the training step (forward with saved activations, backward kernels, Adam) against the
reference golden trace and the oracle's autograd."""
import os

import numpy as np
import pytest
import torch

from oracle import init as oinit
from oracle import loss as oloss
from oracle import net as onet

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), 'golden')


def _net(arch, cout, sd, mode):
    import importlib
    mod = importlib.import_module('segmentation3d.network.' + arch)
    net = mod.SegmentationNet(1, cout)
    net.load_state_dict(sd)
    net.b200_mode = mode
    return net.cuda().train()


@pytest.mark.parametrize('arch,cout,lossname', [('vnet', 2, 'dice'), ('vbnet', 5, 'focal'), ('vnet', 16, 'focal')])
def test_gradients_match_oracle_autograd_fp32(arch, cout, lossname):
    from segmentation3d.loss.focal_loss import FocalLoss
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 5)
    g = torch.Generator().manual_seed(21)
    crops = torch.randn((2, 1, 16, 16, 32), generator=g)
    masks = torch.randint(0, cout, (2, 1, 16, 16, 32), generator=g).float()
    # oracle: torch autograd through the functional restatement
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    probs = onet.forward_with_grad(params, crops)
    if lossname == 'dice':
        ref_loss = oloss.multi_dice_loss(probs, masks, [1.0] * cout)
    else:
        ref_loss = oloss.focal_loss(probs, masks, cout, alpha=[1.0] * cout, gamma=2)
    ref_loss.backward()
    # product
    net = _net(arch, cout, sd, 'fp32')
    out = net(crops.cuda())
    lf = MultiDiceLoss([1.0] * cout, cout, True) if lossname == 'dice' else FocalLoss(cout, alpha=[1.0] * cout, gamma=2, use_gpu=True)
    loss = lf(out, masks.cuda())
    loss.backward()
    assert abs(loss.item() - float(ref_loss)) <= 1e-5
    worst = 0.0
    for name, p in net.named_parameters():
        gr = params[name].grad
        assert p.grad is not None, name
        scale = float(gr.abs().max()) + 1e-12
        err = float((p.grad.cpu() - gr).abs().max()) / scale
        worst = max(worst, err)
        assert err <= 1e-2, (name, err, scale)   # Dice thresholds p > 1/C flip on near-tie voxels: not bit-stable across summation orders
    print(arch, 'worst relative grad error', worst)


def test_train_step_in_the_default_mode_runs_in_bf16(monkeypatch):
    """`seg_train -i cfg` never sets a mode: the default ('auto') and the fp16 / fp32x inference modes must TRAIN in bf16
    (fp16 gradient buffers flush the ~1e-6 data gradients to zero) - network/_graph.py::resolve_mode."""
    from segmentation3d.core.seg_train import make_optimizer, train_step
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    monkeypatch.delenv('SEG3D_MODE', raising=False)
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    g = torch.Generator().manual_seed(5)
    crops = torch.randn((2, 1, 32, 32, 32), generator=g)
    masks = torch.randint(0, 2, (2, 1, 32, 32, 32), generator=g).float()
    ref = float(oloss.multi_dice_loss(onet.forward(sd, crops), masks, [0.5, 0.5]))
    from segmentation3d.network import vnet
    for mode in (None, 'fp16', 'fp32x'):
        net = vnet.SegmentationNet(1, 2)
        net.load_state_dict(sd)
        if mode is not None:
            net.b200_mode = mode
        net = net.cuda().train()
        assert net.b200_mode == (mode or 'auto') and net.resolve_mode(train=True) == 'bf16'
        opt = make_optimizer(net, 1e-4)
        before = [p.detach().clone() for p in net.parameters()]
        loss = train_step(net, opt, MultiDiceLoss([0.5, 0.5], 2, True), crops.cuda(), masks.cuda())
        assert net._plan.mode == 'bf16'
        assert abs(float(loss) - ref) <= 2e-2, (mode, float(loss), ref)
        grads = [p.grad for p in net.parameters()]
        assert all(gr is not None and bool(torch.isfinite(gr).all()) for gr in grads)
        # the deep layers' gradients are the small ones: none of them may have been flushed to zero
        nonzero = [float((gr != 0).float().mean()) for gr in grads]
        assert min(nonzero) > 0.5, min(nonzero)
        assert any(not torch.equal(a, p.detach()) for a, p in zip(before, net.parameters()))
        # inference afterwards runs in the inference mode again, from the updated weights
        net.eval()
        with torch.no_grad():
            net(crops.cuda())
        assert net._plan.mode == ('fp16' if mode in (None, 'fp16') else 'fp32x')


def test_backward_after_a_second_forward_of_the_same_shape_is_refused():
    """the saved activations live in the plan's workspace (one per shape): differentiating a forward whose workspace a later
    forward overwrote must fail loudly, not return the wrong gradients"""
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    net = _net('vnet', 2, oinit.init_state_dict('vnet', 1, 2, 0), 'fp32')
    g = torch.Generator().manual_seed(6)
    a = torch.randn((1, 1, 16, 16, 16), generator=g).cuda()
    m = torch.randint(0, 2, (1, 1, 16, 16, 16), generator=g).float().cuda()
    lf = MultiDiceLoss([0.5, 0.5], 2, True)
    first = lf(net(a), m)
    second = lf(net(a * 0.5), m)
    with pytest.raises(RuntimeError, match='overwritten by a later forward'):
        first.backward()
    second.backward()


def test_two_adam_steps_match_reference_golden():
    """core/seg_train.py:83,119-127 on the golden batch: losses and updated weights of the unmodified reference."""
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    z = np.load(os.path.join(G, 'train_step.npz'))
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    net = _net('vnet', 2, sd, 'fp32')
    g = torch.Generator().manual_seed(21)
    crops = torch.randn((2, 1, 16, 16, 32), generator=g).cuda()
    masks = torch.randint(0, 2, (2, 1, 16, 16, 32), generator=g).float().cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.999))
    lf = MultiDiceLoss([1.0, 1.0], 2, True)
    losses = []
    for _ in range(2):
        opt.zero_grad()
        loss = lf(net(crops), masks)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print('losses', losses, 'reference', z['vnet_dice_losses'])
    assert np.abs(np.array(losses) - z['vnet_dice_losses']).max() <= 2e-4
    got = net.state_dict()
    for k in ('in_block.conv.weight', 'down_64.down_conv.weight', 'up_32.up_conv.weight', 'out_block.conv2.weight',
              'out_block.gn1.weight', 'up_128.up_gn.bias'):
        ref = z['vnet_dice/' + k]
        d = np.abs(got[k].cpu().numpy() - ref)
        # Adam's first steps move every weight by ~lr; a wrong gradient sign shows up as a 2*lr = 2e-4 difference
        assert np.mean(d > 1.5e-4) <= 0.01, (k, float(d.max()), float(np.mean(d > 1.5e-4)))
    gi = net.in_block.conv.weight.grad.cpu().numpy()
    ref = z['vnet_dice_grad_in_block']
    assert np.abs(gi - ref).max() <= 5e-2 * np.abs(ref).max()


def _grad_agreement(ref_grads, net, tag):
    rows = {}
    for name, p in net.named_parameters():
        gr = ref_grads[name].double().flatten()
        gn = p.grad.detach().cpu().double().flatten()
        assert torch.isfinite(gn).all(), name
        nr = float(gr.norm())
        if nr < 1e-10:
            continue
        rows[name] = (float(torch.dot(gr, gn) / (nr * float(gn.norm()) + 1e-300)), float((gr - gn).norm()) / nr)
    worst = min(rows, key=lambda k: rows[k][0])
    print('%s: worst cosine %.5f (%s), worst relative L2 error %.4f' % (tag, rows[worst][0], worst, max(r for _, r in rows.values())))
    return rows


SHALLOW = ('up_64.rblock', 'up_32', 'out_block')


def test_bf16_training_gradients():
    """The training bench runs in bf16 (tensor-core forward, dgrad and wgrad kernels, bf16 activations and data
    gradients, fp32 parameter gradients).  On random-init weights the bf16-rounded program is ill-conditioned below the
    second level: rounding flips ~1 % of the deep ReLU masks, and a 1e-6 relative change of the INPUT moves the
    gradients of the rounded oracle (oracle/reduced_precision.py) itself by 24 % (L2, cosine 0.97) in down_64 ...
    up_128 while the fp32 oracle does not move - measured on the CPU.  So no two bf16 implementations agree
    there better than that; what the kernels must do is (i) reproduce the loss, (ii) stay inside that band against both
    the fp32 oracle's autograd and the rounded oracle's, and (iii) agree tightly where the program is well conditioned:
    the layers next to the loss and the skip path.  The backward itself is pinned stage by stage in
    tests/test_gpu_train_stages.py: every GroupNorm backward, weight gradient, data gradient and the out-block tail of this
    very path, up to the benchmarked 8 x 96^3 step, against float64 recomputed from the buffers each kernel read, to the
    rounding of its own output - weight gradients to the bound their kernels' accumulation length allows, which at 8 x 96^3
    is looser than fp32 (an open finding there) - plus per op: test_gn_bwd_matches_closed_form, test_conv_wgrad_matches_torch,
    and in fp32 above."""
    from oracle import reduced_precision as orp
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, 2, 0), 5)
    g = torch.Generator().manual_seed(33)
    crops = torch.randn((2, 1, 32, 32, 32), generator=g)
    masks = torch.randint(0, 2, (2, 1, 32, 32, 32), generator=g).float()

    def oracle_grads(fwd):
        params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        ref_loss = oloss.multi_dice_loss(fwd(params, crops), masks, [1.0, 1.0])
        ref_loss.backward()
        return float(ref_loss.detach()), {k: p.grad for k, p in params.items()}

    loss32, g32 = oracle_grads(onet.forward_with_grad)
    loss16, g16 = oracle_grads(lambda p, x: orp.forward_with_grad(p, x, torch.bfloat16))
    net = _net('vnet', 2, sd, 'bf16')
    loss = MultiDiceLoss([1.0, 1.0], 2, True)(net(crops.cuda()), masks.cuda())
    loss.backward()
    print('loss: kernels bf16 %.6f, rounded oracle %.6f, fp32 oracle %.6f' % (loss.item(), loss16, loss32))
    assert abs(loss.item() - loss32) <= 2e-3 and abs(loss.item() - loss16) <= 2e-3
    for tag, ref in (('vs bf16-rounded oracle autograd', g16), ('vs fp32 oracle autograd', g32)):
        rows = _grad_agreement(ref, net, tag)
        for name, (cos, rel) in rows.items():
            assert cos >= 0.95 and rel <= 0.35, (tag, name, cos, rel)
            if name.startswith(SHALLOW):
                assert cos >= 0.99 and rel <= 0.15, (tag, name, cos, rel)


def test_adam_step_kernel_matches_torch_adam():
    """seg3d_adam_step against torch.optim.Adam (the reference's optimiser, core/seg_train.py:83) over 4 steps, with and
    without weight decay, on a range whose length is not a multiple of 4"""
    from segmentation3d._b200 import lib as L
    L.load()
    for wd in (0.0, 0.01):
        g = torch.Generator().manual_seed(3)
        n = 100003
        p0 = torch.randn(n, generator=g)
        ref = p0.clone().cuda().requires_grad_(True)
        opt = torch.optim.Adam([ref], lr=1e-3, betas=(0.9, 0.999), weight_decay=wd)
        p = torch.zeros(n + 1, device='cuda')[:n]
        p.copy_(p0)
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        for step in range(1, 5):
            grad = (torch.randn(n, generator=g) * 10 ** float(torch.randint(-6, 1, (1,), generator=g))).cuda()
            ref.grad = grad.clone()
            opt.step()
            L.call('seg3d_adam_step', L.ptr(p), L.ptr(grad), L.ptr(m), L.ptr(v), n, 1e-3, 0.9, 0.999, 1e-8, wd, step, L.stream_ptr())
            torch.cuda.synchronize()
            assert float((p - ref.detach()).abs().max()) <= 2e-6, (wd, step)
        st = opt.state[ref]
        assert float((m - st['exp_avg']).abs().max()) <= 1e-6 * float(st['exp_avg'].abs().max()) + 1e-12
        # (fused multiply-adds round g*g once where torch rounds twice: a few ulp of the largest second moment)
        assert float((v - st['exp_avg_sq']).abs().max()) <= 1e-4 * float(st['exp_avg_sq'].abs().max()) + 1e-20


@pytest.mark.parametrize('arch,cout,mode', [('vnet', 2, 'fp16'), ('vbnet', 5, 'fp32x'), ('vnet', 2, 'fp32'), ('vbnet', 3, 'bf16')])
def test_gather_pack_kernel_reproduces_every_weight_layout(arch, cout, mode):
    """seg3d_gather_pack (one launch, table of index maps) against the per-tensor torch re-layout (plan.py::_Conv.load) for every
    convolution of the network, bit for bit: tensor-core [tap][Cout][Cin], the folded narrow-output layout, split hi / lo
    halves, SIMT [tap][Cin][Cout], transposed convs, zero-padded output channels, biases and GroupNorm affines; and for a
    training plan the flipped / transposed data-gradient weights."""
    import importlib
    mod = importlib.import_module('segmentation3d.network.' + arch)
    net = mod.SegmentationNet(1, cout)
    net.load_state_dict(oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 5))
    net.b200_mode = mode
    net = net.cuda().eval()
    train = mode in ('bf16', 'fp32')
    plan = net._current_plan(train=train)
    assert plan.pack_table is not None and plan._bound_valid()
    with torch.no_grad():
        g = torch.Generator().manual_seed(1)
        for p in net.parameters():
            p.mul_((1.0 + 0.05 * torch.randn(p.shape, generator=g)).cuda())
    sd = {k: v.detach() for k, v in net.state_dict().items()}

    def snapshot(convs):
        out = {}
        for name, c in convs.items():
            out[name] = [t.clone() for t in (c.w, c.w_fold, c.bias) if t is not None]
        return out
    plan.pack_table.run()
    torch.cuda.synchronize()
    fast = snapshot(plan.convs)
    fast_gn = {n: (g_.gamma.clone(), g_.beta.clone()) for n, g_ in plan.gns.items()}
    for c in plan.convs.values():
        c.load(sd)
    slow = snapshot(plan.convs)
    for name in fast:
        for a, b in zip(fast[name], slow[name]):
            assert a.dtype == b.dtype and torch.equal(a, b), (name, mode)
    for n, (ga, be) in fast_gn.items():
        assert torch.equal(ga, sd[n + '.weight']) and torch.equal(be, sd[n + '.bias'])
    if train:
        from segmentation3d._b200.autograd import _Backward
        ws, _ = plan.plan(1, 16, 16, 16, train=True)
        plan._last_sd = sd
        bw = _Backward(plan, ws)
        assert bw.pack_table is not None
        with torch.no_grad():
            for p in net.parameters():
                p.mul_(1.01)
        sd = {k: v.detach() for k, v in net.state_dict().items()}
        plan._last_sd = sd
        bw.pack_table.run()
        torch.cuda.synchronize()
        fast = snapshot(bw.dconv)
        for c in bw.dconv.values():
            c.load(sd)
        slow = snapshot(bw.dconv)
        for name in fast:
            for a, b in zip(fast[name], slow[name]):
                assert torch.equal(a, b), ('dgrad', name, mode)
