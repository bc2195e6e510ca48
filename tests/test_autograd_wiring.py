"""CPU check of the HOST WIRING of the training path (segmentation3d/_b200/autograd.py, loss/_kernels.py) against the
oracle's autograd.

On top of the forward entry points emulated in tests/test_plan_wiring.py, the backward ones are emulated per
include/seg3d_b200.h: seg3d_gn_bwd (both passes, up to three gradient contributions, residual and bias gradients),
seg3d_conv3d_wgrad (kernel weight layouts of the three convolution flavours), seg3d_outblock_tail_bwd (three passes) and the
Dice / focal / cross-entropy reductions.  What runs for real is the backward walk: which gradient buffers feed which unit,
the dgrad convolutions on transformed weights, the flat parameter-gradient buffer and its offsets, the conversion back to
the reference's parameter layouts.  Every parameter gradient of VNet (Dice) and VBNet (focal) must equal the oracle's
autograd gradient; the kernels themselves are pinned by the `-m gpu` tests."""
import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from oracle import loss as oloss
from oracle import net as onet
from test_plan_wiring import _P, _install as _install_forward, _mean_rstd, _rows


def _install(monkeypatch, calls):
    from segmentation3d._b200 import lib
    from segmentation3d.loss import _kernels
    plan = _install_forward(monkeypatch, calls)
    table = {}
    fwd_call = lib.call

    def gn_bwd(dtype, ps, g0, ld0, g1, ld1, g2, ld2, out, out_ld, y, y_ld, C, stats, gamma, beta, eps, sums, dgamma, dbeta,
               dy, dy_ld, dres, dres_ld, dbias, N, nvox, stream):
        g = _rows(g0, N * nvox, ld0, C).double()
        if g1 is not None:
            g = g + _rows(g1, N * nvox, ld1, C).double()
        if g2 is not None:
            g = g + _rows(g2, N * nvox, ld2, C).double()
        mean, rstd = _mean_rstd(stats, float(nvox * C), eps, N)
        yv = _rows(y, N * nvox, y_ld, C).double().view(N, nvox, C)
        xh = (yv - mean) * rstd
        gd = gamma.t.double().view(1, 1, C)
        if out is None:         # ReLU mask recomputed from the raw tensor: fma(y, rstd*gamma, beta - mean*rstd*gamma) > 0
            assert beta is not None and dres is None
            a = (rstd.float() * gamma.t.float().view(1, 1, C)).double()
            b = (beta.t.double().view(1, 1, C) - mean.float().double() * a).float().double()     # one rounding, like the kernel's FFMA
            dz = g.view(N, nvox, C) * ((yv * a + b) > 0)
        else:
            dz = (g * (_rows(out, N * nvox, out_ld, C).double() > 0)).view(N, nvox, C)
        if ps == 0:
            st = sums.t.reshape(-1, 2)
            st[:N, 0] += (dz * gd).flatten(1).sum(1)
            st[:N, 1] += (dz * gd * xh).flatten(1).sum(1)
            dgamma.t.reshape(-1)[dgamma.off:dgamma.off + C] += (dz * xh).sum((0, 1)).float()
            dbeta.t.reshape(-1)[dbeta.off:dbeta.off + C] += dz.sum((0, 1)).float()
        else:
            cnt = float(nvox * C)
            st = sums.t.reshape(-1, 2)
            m1, m2 = (st[:N, 0] / cnt).view(N, 1, 1), (st[:N, 1] / cnt).view(N, 1, 1)
            d = rstd * (gd * dz - m1 - xh * m2)
            dst = _rows(dy, N * nvox, dy_ld, C)
            dst.copy_(d.reshape(-1, C).to(dst.dtype))
            if dres is not None:
                r = _rows(dres, N * nvox, dres_ld, C)
                r.copy_(dz.reshape(-1, C).to(r.dtype))
            if dbias is not None:
                dbias.t.reshape(-1)[dbias.off:dbias.off + C] += d.sum((0, 1)).float()
        calls.append('gn_bwd%d' % ps)
        return 0

    def wgrad(mode, dtype, x, x_ld, Cin, dy, dy_ld, Cout, dw, N, D, H, W, stream):
        xs = _rows(x, N * D * H * W, x_ld, Cin).float().view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        with torch.enable_grad():               # these emulations run inside an autograd backward, where grad mode is off
            if mode == lib.CONV_T2S2:
                w = torch.zeros((Cin, Cout, 2, 2, 2), requires_grad=True)
                y = F.conv_transpose3d(xs, w, None, stride=2)
            else:
                k = 3 if mode == lib.CONV_K3 else 2
                w = torch.zeros((Cout, Cin, k, k, k), requires_grad=True)
                y = F.conv3d(xs, w, None, stride=2 if mode == lib.CONV_K2S2 else 1, padding=1 if mode == lib.CONV_K3 else 0)
            n_out = y.shape[0] * y.shape[2] * y.shape[3] * y.shape[4]
            gy = _rows(dy, n_out, dy_ld, Cout).float().view(y.shape[0], y.shape[2], y.shape[3], y.shape[4], Cout).permute(0, 4, 1, 2, 3)
            y.backward(gy)
        if mode == lib.CONV_T2S2:
            packed = w.grad.permute(0, 2, 3, 4, 1).reshape(-1)                   # [Cin][tap*Cout + co]
        else:
            packed = w.grad.permute(2, 3, 4, 1, 0).reshape(-1)                   # [taps][Cin][Cout]
        dw.t.reshape(-1)[dw.off:dw.off + packed.numel()] += packed
        calls.append('wgrad%d' % mode)
        return 0

    def cin1_wgrad(dtype, xpad, x_pitch, dy, dy_ld, dw, N, D, H, W, stream):
        # the row-padded input of seg3d_conv3d_cin1_fwd; dy must be dense
        assert x_pitch == W + lib.CIN1_PAD and dy_ld == 16
        rows = _rows(xpad, N * D * H, x_pitch, x_pitch)
        xs = rows[:, lib.CIN1_LEFT:lib.CIN1_LEFT + W].contiguous().reshape(-1)
        return wgrad(lib.CONV_K3, dtype, type(xpad)(xs, 0), 1, 1, dy, dy_ld, 16, dw, N, D, H, W, stream)

    def tail_bwd(dtype, ps, y1, ld, C, stats1, g1, b1, w2, bias2, stats2, g2, b2, eps, dprobs, sums2, sums1,
                 dgamma2, dbeta2, dw2, db2, dgamma1, dbeta1, db1, dy1, dy_ld, N, nvox, stream):
        if ps != 2:                 # every output is produced in the last pass here; the sums are internal to the kernel
            calls.append('tail_bwd%d' % ps)
            return 0
        with torch.enable_grad():
            y = _rows(y1, N * nvox, ld, C).float().view(N, nvox, C).clone().requires_grad_(True)
            leaves = [t.t.float().reshape(-1)[t.off:t.off + n].clone().requires_grad_(True)
                      for t, n in ((g1, C), (b1, C), (w2, C * C), (bias2, C), (g2, C), (b2, C))]
            G1, B1, W2, BI2, G2, B2 = leaves
            a = F.relu(F.group_norm(y.permute(0, 2, 1), 1, G1, B1, eps))                  # [N, C, nvox]
            z = torch.einsum('oc,ncv->nov', W2.view(C, C), a) + BI2.view(1, C, 1)
            p = F.softmax(F.group_norm(z, 1, G2, B2, eps), 1)
            p.backward(dprobs.t.float().reshape(N, C, nvox))
        for dst, src in ((dgamma1, G1), (dbeta1, B1), (dw2, W2), (db2, BI2), (dgamma2, G2), (dbeta2, B2)):
            dst.t.reshape(-1)[dst.off:dst.off + src.numel()] += src.grad
        db1.t.reshape(-1)[db1.off:db1.off + C] += y.grad.sum((0, 1))
        d = _rows(dy1, N * nvox, dy_ld, C)
        d.copy_(y.grad.reshape(-1, C).to(d.dtype))
        calls.append('tail_bwd2')
        return 0

    def dice_terms(probs, target, B, C, n, terms, stream):
        p = probs.t.float().reshape(B, C, n)
        t = target.t.float().reshape(B, n)
        for c in range(C):
            q = p[:, c] * (p[:, c] > 1.0 / C)
            tv = (t == c).float()
            terms.t[:, c, 0] += (q * tv).double().sum(1)
            terms.t[:, c, 1] += (q * q).double().sum(1)
            terms.t[:, c, 2] += tv.double().sum(1)
        return 0

    def dice_bwd(probs, target, B, C, n, coef, grad, stream):
        p = probs.t.float().reshape(B, C, n)
        t = target.t.float().reshape(B, n)
        cf = coef.t.float().reshape(B, C, 2)
        g = torch.zeros_like(p)
        for c in range(C):
            m = (p[:, c] > 1.0 / C).float()
            g[:, c] = m * (cf[:, c, 0:1] * (t == c).float() + cf[:, c, 1:2] * p[:, c])
        grad.t.copy_(g.reshape(grad.t.shape))
        return 0

    def focal_fwd(probs, target, B, C, n, alpha, gamma, partial, stream):
        p = probs.t.float().reshape(B, C, n)
        t = target.t.float().reshape(B, n).long()
        pt = p.gather(1, t.unsqueeze(1))[:, 0] + 1e-10
        partial.t[0] += (-alpha.t.float().reshape(-1)[t] * (1 - pt) ** gamma * torch.log(pt)).double().sum()
        return 0

    def focal_bwd(probs, target, B, C, n, alpha, gamma, scale, grad, stream):
        p = probs.t.float().reshape(B, C, n)
        t = target.t.float().reshape(B, n).long()
        pt = p.gather(1, t.unsqueeze(1))[:, 0] + 1e-10
        a = alpha.t.float().reshape(-1)[t]
        om = 1 - pt
        g = a * (gamma * om ** (gamma - 1) * torch.log(pt) - om ** gamma / pt) if gamma > 0 else -a / pt
        out = torch.zeros_like(p)
        out.scatter_(1, t.unsqueeze(1), (g * scale).unsqueeze(1))
        grad.t.copy_(out.reshape(grad.t.shape))
        return 0

    def adam_step(param, grad, m, v, n, lr, b1, b2, eps, wd, step, stream):
        """torch/optim/adam.py::_single_tensor_adam on flat ranges"""
        p_, g_, m_, v_ = (t.flat()[:n] for t in (param, grad, m, v))
        g = g_ + wd * p_ if wd else g_.clone()
        m_.lerp_(g, 1 - b1)
        v_.mul_(b2).addcmul_(g, g, value=1 - b2)
        denom = (v_.sqrt() / (1 - b2 ** step) ** 0.5).add_(eps)
        p_.addcdiv_(m_, denom, value=-lr / (1 - b1 ** step))
        calls.append('adam_step')
        return 0

    def _ce_terms(x, t, B, C, n, w, ignore_index):
        xs = x.t.float().reshape(B, C, n).double()
        tt = t.t.float().reshape(B, n).long()
        valid = tt != ignore_index
        tc = tt.clamp(0, C - 1)
        wt = (w.t.double().reshape(-1)[tc] if w is not None else torch.ones_like(xs[:, 0])) * valid
        return xs, tc, wt

    def ce_fwd(x, t, B, C, n, w, ignore_index, part, lmap, stream):
        xs, tc, wt = _ce_terms(x, t, B, C, n, w, ignore_index)
        loss = wt * (torch.logsumexp(xs, 1) - xs.gather(1, tc.unsqueeze(1))[:, 0])
        part.t[0] += loss.sum()
        part.t[1] += wt.sum()
        if lmap is not None:
            lmap.t.copy_(loss.reshape(lmap.t.shape).float())
        return 0

    def ce_bwd(x, t, B, C, n, w, ignore_index, scale, gmap, grad, stream):
        xs, tc, wt = _ce_terms(x, t, B, C, n, w, ignore_index)
        g = torch.softmax(xs, 1)
        g.scatter_add_(1, tc.unsqueeze(1), -torch.ones_like(xs[:, :1]))
        g = g * (wt * (gmap.t.double().reshape(B, n) if gmap is not None else scale)).unsqueeze(1)
        grad.t.copy_(g.reshape(grad.t.shape).float())
        return 0

    table.update({'seg3d_adam_step': adam_step, 'seg3d_ce_fwd': ce_fwd, 'seg3d_ce_bwd': ce_bwd})
    table.update({'seg3d_gn_bwd': gn_bwd, 'seg3d_conv3d_wgrad': wgrad, 'seg3d_conv3d_cin1_wgrad': cin1_wgrad, 'seg3d_outblock_tail_bwd': tail_bwd,
                  'seg3d_dice_terms': dice_terms, 'seg3d_dice_bwd': dice_bwd, 'seg3d_focal_fwd': focal_fwd, 'seg3d_focal_bwd': focal_bwd})
    monkeypatch.setattr(lib, 'call', lambda name, *a: table[name](*a) if name in table else fwd_call(name, *a))

    def check(probs, target):
        B, C = probs.shape[0], probs.shape[1]
        n = probs[0, 0].numel()
        assert target.numel() == B * n
        return B, C, n
    monkeypatch.setattr(_kernels, '_check', check)
    return plan


@pytest.mark.parametrize('arch,cout,lossname,mode', [('vnet', 2, 'dice', 'fp32'), ('vbnet', 5, 'focal', 'fp32'), ('vnet', 2, 'dice', 'bf16')])
def test_backward_walk_reproduces_oracle_autograd(monkeypatch, arch, cout, lossname, mode):
    import importlib
    from segmentation3d.loss.focal_loss import FocalLoss
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    calls = []
    _install(monkeypatch, calls)
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 5)
    g = torch.Generator().manual_seed(21)
    crops = torch.randn((2, 1, 16, 16, 32), generator=g)
    masks = torch.randint(0, cout, (2, 1, 16, 16, 32), generator=g).float()
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    probs = onet.forward_with_grad(params, crops)
    ref_loss = oloss.multi_dice_loss(probs, masks, [1.0] * cout) if lossname == 'dice' else \
        oloss.focal_loss(probs, masks, cout, alpha=[1.0] * cout, gamma=2)
    ref_loss.backward()

    net = importlib.import_module('segmentation3d.network.' + arch).SegmentationNet(1, cout)
    net.load_state_dict(sd)
    net.b200_mode = mode
    net.train()
    lf = MultiDiceLoss([1.0] * cout, cout, False) if lossname == 'dice' else FocalLoss(cout, alpha=[1.0] * cout, gamma=2, use_gpu=False)
    for step in range(2):                       # the second step reuses the cached plan and backward state (refresh paths)
        net.zero_grad()
        loss = lf(net(crops), masks)
        loss.backward()
    tol_loss, tol = (1e-5, 1e-2) if mode == 'fp32' else (5e-3, None)   # 1e-2: Dice thresholds flip on near-tie voxels (as in tests/test_gpu_train.py)
    assert abs(loss.item() - float(ref_loss.detach())) <= tol_loss
    worst = 0.0
    for name, p in net.named_parameters():
        gr = params[name].grad
        assert p.grad is not None and p.grad.shape == gr.shape, name
        if tol is not None:
            err = float((p.grad - gr).abs().max()) / (float(gr.abs().max()) + 1e-12)
            worst = max(worst, err)
            assert err <= tol, (name, err)
        else:                                   # bf16 storage: direction only (tests/test_gpu_train.py explains the band)
            a, b = gr.double().flatten(), p.grad.double().flatten()
            if float(a.norm()) > 1e-10:
                assert float(torch.dot(a, b) / (a.norm() * b.norm())) >= 0.9, name
    n_units = sum(1 for k, v in sd.items() if k.endswith('.weight') and v.dim() == 5) - 2      # conv1 / conv2 of the out block
    assert calls.count('gn_bwd0') == calls.count('gn_bwd1') == 2 * n_units
    assert calls.count('tail_bwd2') == 2


def test_one_launch_repack_unpack_and_flat_adam_match_the_torch_path(monkeypatch):
    """_b200/packing.py + _b200/optim.py: with the parameters bound to the plan, a training step re-packs every forward and
    data-gradient weight with one seg3d_gather_pack launch, un-packs the weight gradients with another, and updates all
    parameters with one seg3d_adam_step - the same numbers as the per-tensor torch path (SEG3D_PACK_KERNEL=0 + torch Adam)."""
    from segmentation3d.core.seg_train import make_optimizer, train_step
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    import contextlib
    import importlib
    from segmentation3d._b200.optim import FlatAdam
    monkeypatch.setattr(FlatAdam, '_on_device', staticmethod(lambda p: True))
    monkeypatch.setattr(torch.cuda, 'device', lambda d: contextlib.nullcontext())
    results = {}
    for arch, cout, mode in (('vnet', 2, 'bf16'), ('vbnet', 3, 'fp32')):
        for fast in (True, False):
            calls = []
            _install(monkeypatch, calls)
            monkeypatch.setenv('SEG3D_PACK_KERNEL', '1' if fast else '0')
            mod = importlib.import_module('segmentation3d.network.' + arch)
            torch.manual_seed(0)
            net = mod.SegmentationNet(1, cout)
            net.load_state_dict(oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 3))
            net.b200_mode = mode
            net.train()
            opt = make_optimizer(net, 1e-3) if fast else torch.optim.Adam(net.parameters(), lr=1e-3)
            g = torch.Generator().manual_seed(9)
            crops = torch.randn((2, 1, 16, 16, 16), generator=g)
            masks = torch.randint(0, cout, (2, 1, 16, 16, 16), generator=g).float()
            lf = MultiDiceLoss([1.0] * cout, cout, False)
            losses = [float(train_step(net, opt, lf, crops, masks)) for _ in range(3)]
            if fast:
                assert calls.count('adam_step') == 3 and opt.used_flat_grads
                st = opt.state_dict()['state']
                assert len(st) == len(list(net.parameters())) and float(st[0]['step']) == 3.0
                assert st[0]['exp_avg'].shape == net.in_block.conv.weight.shape
            results[(arch, fast)] = (losses, [p.detach().clone() for p in net.parameters()])
        (la, pa), (lb, pb) = results[(arch, True)], results[(arch, False)]
        assert max(abs(a - b) for a, b in zip(la, lb)) <= 1e-5, (arch, la, lb)
        worst = max(float((a - b).abs().max()) for a, b in zip(pa, pb))
        assert worst <= 2e-5, (arch, worst)        # three Adam steps of size 1e-3: identical update rule, fp32 rounding apart
