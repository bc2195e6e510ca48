"""CPU check of the whole network's partial backward (segmentation3d/_b200/autograd.py::_Backward.schedule, network/_graph.py,
_b200/optim.py) with the C-ABI entry points emulated as in tests/test_autograd_wiring.py.

* An all-trainable step with an input that does not require grad issues exactly the launches (entry names and scalar
  arguments) of the parent commit's backward: tests/golden/backward_launches_all_trainable.json, written by running this
  file as a script (`python tests/test_partial_backward_wiring.py`) on that commit.
* Freeze masks: every requested gradient (the input gradient included) equals the oracle's autograd, frozen parameters
  get None, and the launch counts follow the schedule rule, derived here from the network's topology: in a V-shaped net
  every conv unit's input window holds the output of the unit before it in forward order, so unit i is needed exactly
  when the input needs a gradient or a parameter of units 0..i is trainable.
* FlatAdam skips parameters without a gradient, as torch.optim.Adam does.
* Data parallel: only the trainable slots of the flat gradient buffer are all-reduced."""
import json
import os
import random
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(HERE, '..', 'medical-segmentation3d-toolkit_b200'), os.path.join(HERE, '..'), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from oracle import init as oinit  # noqa: E402
from oracle import loss as oloss  # noqa: E402
from oracle import net as onet  # noqa: E402
from test_autograd_wiring import _install as _install_train  # noqa: E402
from test_plan_wiring import _P, _rows  # noqa: E402

GOLDEN = os.path.join(HERE, 'golden', 'backward_launches_all_trainable.json')
CASES = [('vnet', 2, 'bf16'), ('vnet', 2, 'fp32'), ('vbnet', 3, 'bf16'), ('vbnet', 3, 'fp32')]
SHAPE = (2, 1, 16, 16, 32)
SMALL = (1, 1, 16, 16, 16)          # the freeze-mask sweep: many steps, the smallest VNet input


def _install(monkeypatch, calls):
    """the training emulation plus the two new entry points; returns the list every lib.call appends
    [name, scalar arguments...] to (pointers as 'p', NULL as None)"""
    import torch.nn.functional as F
    from segmentation3d._b200 import lib
    _install_train(monkeypatch, calls)
    inner = lib.call
    launches = []

    def cin1_dgrad(dtype, gy, ld, w, dx, N, D, H, W, stream):
        g = _rows(gy, N * D * H * W, ld, 16).float().view(N, D, H, W, 16).permute(0, 4, 1, 2, 3)
        wk = w.t.float().reshape(-1)[w.off:w.off + 27 * 16].view(3, 3, 3, 16).permute(3, 0, 1, 2).unsqueeze(1)   # [16,1,3,3,3]
        dx.t.reshape(-1)[dx.off:dx.off + N * D * H * W].copy_(F.conv_transpose3d(g, wk, padding=1).reshape(-1))
        calls.append('cin1_dgrad')
        return 0

    def adam_ranges(param, grad, m, v, table, n_ranges, lr, b1, b2, eps, wd, stream):
        for e in table[:n_ranges]:
            o, n, step = int(e.offset), int(e.n), int(e.step)
            p_, g_, m_, v_ = (t.flat()[o:o + n] for t in (param, grad, m, v))
            g = g_ + wd * p_ if wd else g_.clone()
            m_.lerp_(g, 1 - b1)
            v_.mul_(b2).addcmul_(g, g, value=1 - b2)
            denom = (v_.sqrt() / (1 - b2 ** step) ** 0.5).add_(eps)
            p_.addcdiv_(m_, denom, value=-lr / (1 - b1 ** step))
        calls.append('adam_ranges')
        return 0

    def grad_to_ncdhw(dtype, n, g0, ld0, off0, g1, ld1, off1, g2, ld2, off2, C, N, nvox, out, stream):
        acc = torch.zeros((N * nvox, C), dtype=torch.float32)
        for g, ld, off in ((g0, ld0, off0), (g1, ld1, off1), (g2, ld2, off2))[:n]:
            assert ld >= off + C and g.t.dtype == lib.TORCH_DTYPE[dtype]
            acc += _rows(_P(g.t, g.off + off), N * nvox, ld, C).float()
        out.t.reshape(-1)[out.off:out.off + N * C * nvox].copy_(acc.view(N, nvox, C).permute(0, 2, 1).reshape(-1))
        return 0

    extra = {'seg3d_conv3d_cin1_dgrad': cin1_dgrad, 'seg3d_adam_step_ranges': adam_ranges, 'seg3d_grad_to_ncdhw': grad_to_ncdhw}

    def call(name, *a):
        launches.append([name] + [x if isinstance(x, (int, float)) or x is None else 'p' for x in a])
        return extra[name](*a) if name in extra else inner(name, *a)
    monkeypatch.setattr(lib, 'call', call)
    return launches


def _net(arch, cout, mode, sd, cin=1):
    import importlib
    net = importlib.import_module('segmentation3d.network.' + arch).SegmentationNet(cin, cout)
    net.load_state_dict(sd)
    net.b200_mode = mode
    net.train()
    return net


def _data(cout, shape=SHAPE):
    g = torch.Generator().manual_seed(21)
    crops = torch.randn(shape, generator=g)
    masks = torch.randint(0, cout, shape, generator=g).float()
    return crops, masks


def record_backward(monkeypatch, arch, cout, mode):
    """launch list of the backward of an all-trainable Dice step, input not requiring grad (the second step: cached state)"""
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    launches = _install(monkeypatch, [])
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 5)
    net = _net(arch, cout, mode, sd)
    crops, masks = _data(cout)
    lf = MultiDiceLoss([1.0] * cout, cout, False)
    for _ in range(2):
        net.zero_grad()
        loss = lf(net(crops), masks)
        del launches[:]
        loss.backward()
    return list(launches)


@pytest.mark.parametrize('arch,cout,mode', CASES)
def test_all_trainable_backward_issues_the_parent_launches(monkeypatch, arch, cout, mode):
    golden = json.load(open(GOLDEN))['%s_%d_%s' % (arch, cout, mode)]
    got = json.loads(json.dumps(record_backward(monkeypatch, arch, cout, mode)))
    assert got == golden


# ---- freeze masks ---------------------------------------------------------------------------------------------------------
def _unit_convs(net):
    """conv names of the walked units in forward order (every 5-D conv weight but the out block's)"""
    return [n[:-len('.weight')] for n, p in net.named_parameters() if p.dim() == 5 and not n.startswith('out_block')]


def _unit_params(conv):
    gn = conv[:-len('_conv')] + '_gn' if conv.endswith('_conv') else conv[:-len('conv')] + 'gn'
    return [conv + '.weight', conv + '.bias', gn + '.weight', gn + '.bias']


def _expected_counts(net, need, need_input):
    convs = _unit_convs(net)
    n_gn = n_w = n_d = 0
    upstream = need_input
    prev_needed = need_input
    for c in convs:
        pars = _unit_params(c)
        upstream = upstream or any(p in need for p in pars)
        if upstream:
            n_gn += 2
            n_w += int(pars[0] in need or pars[1] in need)
            n_d += int(prev_needed) if c != 'in_block.conv' else 0
        prev_needed = upstream
    tail = upstream or any(n.startswith('out_block') for n in need)
    tail_w = 'out_block.conv1.weight' in need or 'out_block.conv1.bias' in need
    return {'seg3d_gn_bwd': n_gn, 'wgrad': n_w + int(tail_w), 'seg3d_conv3d_fwd': n_d + int(upstream),
            'seg3d_outblock_tail_bwd': 3 if tail else 0, 'seg3d_conv3d_cin1_dgrad': int(need_input)}


def _masks(names):
    enc = [n for n in names if n.startswith(('in_block', 'down_'))]
    out = [
        ('encoder_frozen', [n for n in names if n not in enc], False),
        ('decoder_frozen', [n for n in names if not n.startswith('up_')], False),
        ('only_out_block', [n for n in names if n.startswith('out_block')], False),
        ('only_in_block', [n for n in names if n.startswith('in_block')], False),
        ('all_frozen_input', [], True),
        ('all_trainable_input', list(names), True),
    ]
    for s in range(5):
        r = random.Random(100 + s)
        out.append(('random%d' % s, [n for n in names if r.random() < 0.5], r.random() < 0.5))
    return out


_ORACLE = {}


def _oracle(arch, cout, sd):
    if arch not in _ORACLE:
        crops, masks = _data(cout, SMALL)
        params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        x = crops.clone().requires_grad_(True)
        oloss.multi_dice_loss(onet.forward_with_grad(params, x), masks, [1.0] * cout).backward()
        _ORACLE[arch] = ({k: v.grad for k, v in params.items()}, x.grad)
    return _ORACLE[arch]


def _close(got, ref, mode, what):
    assert got is not None and got.shape == ref.shape, what
    if mode == 'fp32':      # 1e-2: Dice thresholds flip on near-tie voxels (tests/test_autograd_wiring.py)
        err = float((got - ref).abs().max()) / (float(ref.abs().max()) + 1e-12)
        assert err <= 1e-2, (what, err)
    else:                   # bf16 storage: direction only (tests/test_autograd_wiring.py)
        a, b = ref.double().flatten(), got.double().flatten()
        if float(a.norm()) > 1e-10:
            assert float(torch.dot(a, b) / (a.norm() * b.norm())) >= 0.9, what


@pytest.mark.parametrize('arch,cout,mode', [('vnet', 2, 'fp32'), ('vnet', 2, 'bf16'), ('vbnet', 3, 'fp32')])
def test_freeze_masks_match_oracle_and_skip_launches(monkeypatch, arch, cout, mode):
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    launches = _install(monkeypatch, [])
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 5)
    ref_g, ref_x = _oracle(arch, cout, sd)
    net = _net(arch, cout, mode, sd)
    names = [n for n, _ in net.named_parameters()]
    crops, masks = _data(cout, SMALL)
    lf = MultiDiceLoss([1.0] * cout, cout, False)
    for label, need, need_input in _masks(names):
        need = set(need)
        for n, p in net.named_parameters():
            p.requires_grad_(n in need)
            p.grad = None
        x = crops.clone().requires_grad_(need_input)
        loss = lf(net(x), masks)
        del launches[:]
        loss.backward()
        for n, p in net.named_parameters():
            if n in need:
                _close(p.grad, ref_g[n], mode, (label, n))
            else:
                assert p.grad is None, (label, n)
        if need_input:
            _close(x.grad, ref_x, mode, (label, 'input'))
        else:
            assert x.grad is None
        want = _expected_counts(net, need, need_input)
        names_l = [e[0] for e in launches]
        got = {k: names_l.count(k) for k in want if k != 'wgrad'}
        got['wgrad'] = names_l.count('seg3d_conv3d_wgrad') + names_l.count('seg3d_conv3d_cin1_wgrad')
        assert got == want, (label, got, want)


def test_input_requiring_grad_alone_runs_the_training_path(monkeypatch):
    """network/_graph.py: with every parameter frozen, an input that requires grad still gets a differentiable output"""
    _install(monkeypatch, [])
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, 2, 0), 5)
    net = _net('vnet', 2, 'fp32', sd)
    for p in net.parameters():
        p.requires_grad_(False)
    crops, _ = _data(2, SMALL)
    assert net(crops).grad_fn is None
    y = net(crops.clone().requires_grad_(True))
    assert y.grad_fn is not None
    with torch.no_grad():
        assert net(crops.clone().requires_grad_(True)).grad_fn is None


@pytest.mark.parametrize('mode', ['fp32', 'bf16'])
def test_multi_channel_input_gradient(monkeypatch, mode):
    """in_channels > 1: the input gradient takes the generic data-gradient convolution + seg3d_grad_to_ncdhw, built only
    once a step asks for it"""
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    launches = _install(monkeypatch, [])
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 2, 2, 0), 5)
    g = torch.Generator().manual_seed(22)
    crops = torch.randn((1, 2, 16, 16, 16), generator=g)
    masks = torch.randint(0, 2, (1, 1, 16, 16, 16), generator=g).float()
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xr = crops.clone().requires_grad_(True)
    oloss.multi_dice_loss(onet.forward_with_grad(params, xr), masks, [1.0, 1.0]).backward()
    net = _net('vnet', 2, mode, sd, cin=2)
    lf = MultiDiceLoss([1.0, 1.0], 2, False)
    for label, trainable, need_input in (('params', True, False), ('input_only', False, True), ('both', True, True)):
        for p in net.parameters():
            p.requires_grad_(trainable)
            p.grad = None
        x = crops.clone().requires_grad_(need_input)
        loss = lf(net(x), masks)
        del launches[:]
        loss.backward()
        bw = net._plan._plans[(1, 16, 16, 16, True)][0]['bwd']
        names_l = [e[0] for e in launches]
        assert names_l.count('seg3d_grad_to_ncdhw') == int(need_input), label
        if label == 'params':
            assert bw.dconv_in is None and bw.gd_in is None         # nothing built for an input gradient nobody asked for
            assert x.grad is None
        else:
            _close(x.grad, xr.grad, mode, (label, 'input'))
        for n, p in net.named_parameters():
            if trainable:
                _close(p.grad, params[n].grad, mode, (label, n))
            else:
                assert p.grad is None, (label, n)


# ---- FlatAdam --------------------------------------------------------------------------------------------------------------
def _adam_params(seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(s, generator=g).requires_grad_(True) for s in ((7, 3), (5,), (4, 4, 2), (3,), (6, 1))]


def test_flat_adam_skips_parameters_without_gradient_like_torch(monkeypatch):
    import contextlib
    from segmentation3d._b200.optim import FlatAdam
    calls = []
    launches = _install(monkeypatch, calls)
    monkeypatch.setattr(FlatAdam, '_on_device', staticmethod(lambda p: True))
    monkeypatch.setattr(torch.cuda, 'device', lambda d: contextlib.nullcontext())
    ours, ref = _adam_params(0), _adam_params(0)
    opt = FlatAdam(ours, lr=1e-2, weight_decay=1e-3)
    topt = torch.optim.Adam(ref, lr=1e-2, weight_decay=1e-3)
    frozen = {1, 3}
    g = torch.Generator().manual_seed(1)
    for step in range(1, 6):
        held = {i: (ours[i].detach().clone(), opt.state[ours[i]]['exp_avg'].clone() if ours[i] in opt.state and 'exp_avg' in opt.state[ours[i]] else None)
                for i in frozen} if step <= 2 else {}
        for i, (a, b) in enumerate(zip(ours, ref)):
            gr = torch.randn(a.shape, generator=g)
            a.grad = None if (step <= 2 and i in frozen) else gr.clone()
            b.grad = None if (step <= 2 and i in frozen) else gr.clone()
        del launches[:]
        opt.step()
        topt.step()
        assert [e[0] for e in launches] == ['seg3d_adam_step_ranges']
        for i, (a, b) in enumerate(zip(ours, ref)):
            assert float((a - b).detach().abs().max()) <= 1e-7 * float(b.detach().abs().max()), (step, i)
            if b in topt.state:
                for k in ('exp_avg', 'exp_avg_sq'):
                    rm, om = topt.state[b][k], opt.state[a][k]
                    assert float((om - rm).abs().max()) <= 1e-7 * (float(rm.abs().max()) + 1e-30), (step, i, k)
                assert float(opt.state[a]['step']) == float(topt.state[b]['step'])
        for i, (p0, m0) in held.items():
            assert torch.equal(ours[i].detach(), p0), (step, i)
            assert float(opt.state[ours[i]]['step']) == 0.0
            if m0 is not None:
                assert torch.equal(opt.state[ours[i]]['exp_avg'], m0)


def test_flat_adam_with_every_gradient_issues_one_launch(monkeypatch):
    import contextlib
    from segmentation3d._b200.optim import FlatAdam
    launches = _install(monkeypatch, [])
    monkeypatch.setattr(FlatAdam, '_on_device', staticmethod(lambda p: True))
    monkeypatch.setattr(torch.cuda, 'device', lambda d: contextlib.nullcontext())
    ours = _adam_params(2)
    opt = FlatAdam(ours, lr=1e-3)
    for step in range(1, 4):
        for p in ours:
            p.grad = torch.ones_like(p)
        del launches[:]
        opt.step()
        total = opt._flat[4]
        assert launches == [['seg3d_adam_step', 'p', 'p', 'p', 'p', total, 1e-3, 0.9, 0.999, 1e-8, 0.0, step, 0]]
    assert len({id(opt.state[p]['step']) for p in ours}) == len(ours)      # one step tensor per parameter


# ---- data parallel ---------------------------------------------------------------------------------------------------------
def _ddp_worker(rank, world, port, q):
    import torch.distributed as dist
    for p in (os.path.join(HERE, '..', 'medical-segmentation3d-toolkit_b200'), os.path.join(HERE, '..'), HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    from test_dist_gloo import _Patch
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    os.environ['SEG3D_ALLREDUCE_BUCKET_MB'] = '1'
    _install(_Patch(), [])
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, 2, 0), 5)
    net = _net('vnet', 2, 'fp32', sd)
    enc = ('in_block', 'down_32', 'down_64')
    for n, p in net.named_parameters():
        p.requires_grad_(not n.startswith(enc))
    crops, masks = _data(2)
    real = dist.all_reduce
    spans = []

    def all_reduce(t, *a, **k):
        spans.append((t.storage_offset(), t.storage_offset() + t.numel()))
        return real(t, *a, **k)
    dist.all_reduce = all_reduce
    loss = MultiDiceLoss([1.0, 1.0], 2, False)(net(crops[rank:rank + 1]), masks[rank:rank + 1])
    loss.backward()
    bw = net._plan._plans[(1,) + SHAPE[2:] + (True,)][0]['bwd']
    trainable = [n for n, p in net.named_parameters() if p.requires_grad]
    lo = min(bw.pg_off[n] for n in trainable)
    hi = max(bw.pg_off[n] + bw.pgrad[n].numel() for n in trainable)
    frozen_none = all(p.grad is None for p in net.parameters() if not p.requires_grad)
    grads = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
    got = [None] * world
    dist.all_gather_object(got, grads)
    same = all(torch.equal(got[0][n], got[1][n]) for n in got[0])
    q.put((rank, sorted(spans), lo, hi, frozen_none, same, net._plan.grads_reduced_in_backward))
    dist.destroy_process_group()


def test_data_parallel_all_reduce_covers_exactly_the_trainable_slots():
    import torch.multiprocessing as mp
    from test_dist_gloo import _free_port
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, spans, lo, hi, frozen_none, same, reduced in res:
        assert reduced and frozen_none and same, rank
        assert len(spans) > 1, 'the bucketed all-reduce should run in several pieces'
        assert spans[0][0] == lo and spans[-1][1] == hi, (spans[0], spans[-1], lo, hi)
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:])), spans     # contiguous, no gaps, no overlap


if __name__ == '__main__':
    # writes the golden launch lists; run on the parent commit's tree with its own tests/ on the path
    mp_ = pytest.MonkeyPatch()
    out = {}
    for arch, cout, mode in CASES:
        out['%s_%d_%s' % (arch, cout, mode)] = record_backward(mp_, arch, cout, mode)
        mp_.undo()
    with open(sys.argv[1] if len(sys.argv) > 1 else GOLDEN, 'w') as f:
        json.dump(out, f, indent=0)
