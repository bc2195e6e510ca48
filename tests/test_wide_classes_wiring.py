"""CPU check of the plan's wiring for nets with more than 16 classes (the tensor-core tail, csrc/tail_wide.cu).

The emulation table of test_plan_wiring._install is extended with seg3d_outblock_tail_wide (include/seg3d_b200.h: fp32
raw rows of pitch ld, only channels < C read; pass 0 accumulates the GN2 sums, pass 1 writes probs[n][c][v]) by wrapping
lib.call.  What runs for real is the plan: the padded out_block.conv1, its fp32 raw buffer and pitch, the two tail launches,
for VNet and VBNet in every execution mode; up to 16 classes the launch list must stay the existing one."""
import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from oracle import net as onet
from test_plan_wiring import _install as _install_forward, _mean_rstd, _rows, _stat_rows

TOL = {'fp32': 2e-5, 'fp16': 2e-2, 'bf16': 1.5e-1, 'fp32x': 1e-4}


def _install(monkeypatch, calls):
    plan = _install_forward(monkeypatch, calls)
    lib = plan.lib
    forward_call = lib.call

    def tail_wide(ps, y1, ld, C, stats1, g1, b1, w2, bias2, eps, stats2, g2, b2, probs, N, nvox, stream):
        assert ps in (0, 1) and 1 <= C <= 127 and ld >= C and ld % 4 == 0
        assert y1.t.dtype == torch.float32
        ys = _rows(y1, N * nvox, ld, C).float().view(N, nvox, C)
        mean, rstd = _mean_rstd(stats1, float(nvox * C), eps, N)
        h = F.relu(((ys.double() - mean) * rstd).float() * g1.t.view(1, 1, C) + b1.t.view(1, 1, C))
        z = h @ w2.t.view(C, C).t() + bias2.t.view(1, 1, C)
        if ps == 0:
            rows = _stat_rows(stats2, N)
            rows[:, 0] += z.double().flatten(1).sum(1)
            rows[:, 1] += (z.double() ** 2).flatten(1).sum(1)
        else:
            mean, rstd = _mean_rstd(stats2, float(nvox * C), eps, N)
            z = ((z.double() - mean) * rstd).float() * g2.t.view(1, 1, C) + b2.t.view(1, 1, C)
            probs.t.reshape(-1)[probs.off:probs.off + N * C * nvox].copy_(F.softmax(z, 2).permute(0, 2, 1).reshape(-1))
        calls.append('tail_wide%d' % ps)
        return 0

    def call(name, *args):
        if name == 'seg3d_outblock_tail_wide':
            return tail_wide(*args)
        return forward_call(name, *args)

    monkeypatch.setattr(lib, 'call', call)
    return plan


@pytest.mark.parametrize('arch,cout', [('vnet', 17), ('vbnet', 32), ('vnet', 127)])
@pytest.mark.parametrize('mode', ['fp32', 'fp16', 'bf16', 'fp32x'])
def test_wide_net_issues_the_tensor_core_tail(monkeypatch, arch, cout, mode):
    calls = []
    plan = _install(monkeypatch, calls)
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 11)
    x = torch.randn((2, 1, 16, 32, 16), generator=torch.Generator().manual_seed(6))
    ref = onet.forward(sd, x)
    p = plan.NetPlan(sd, mode=mode, device='cpu')
    got = p.forward(x).clone()
    assert got.shape == ref.shape == (2, cout, 16, 32, 16)
    err = float((got - ref).abs().max())
    assert err <= TOL[mode], (arch, cout, mode, err)
    assert float((got.sum(1) - 1).abs().max()) <= 1e-5
    assert calls[-2:] == ['tail_wide0', 'tail_wide1']
    assert 'tail_stats' not in calls and 'tail_probs' not in calls
    ws, _ = p.plan(2, 16, 32, 16)
    cp = (cout + 15) // 16 * 16
    raw = ws['tail']['raw']
    assert raw.buf.dtype == torch.float32 and raw.ld == cp
    c1 = p.convs['out_block.conv1']
    assert c1.cout == (cout if mode == 'fp32' else cp)                # zero-padded to Cp on the tensor cores
    kinds = [m['kind'] for m in ws['meta'] if m['name'].startswith('out_block.tail')]
    assert kinds == ['tail_wide', 'tail_wide']


@pytest.mark.parametrize('arch,cout', [('vnet', 2), ('vbnet', 5), ('vnet', 16)])
@pytest.mark.parametrize('mode', ['fp32', 'fp16', 'bf16', 'fp32x'])
def test_up_to_sixteen_classes_keep_the_simt_tail(monkeypatch, arch, cout, mode):
    calls = []
    plan = _install(monkeypatch, calls)
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 3)
    x = torch.randn((1, 1, 16, 16, 32), generator=torch.Generator().manual_seed(2))
    p = plan.NetPlan(sd, mode=mode, device='cpu')
    got = p.forward(x)
    assert float((got - onet.forward(sd, x)).abs().max()) <= TOL[mode]
    assert not p.wide
    assert calls[-2:] == ['tail_stats', 'tail_probs'] and not any(c.startswith('tail_wide') for c in calls)
    ws, _ = p.plan(1, 16, 16, 32)
    assert [m['kind'] for m in ws['meta'] if m['name'].startswith('out_block.tail')] == ['tail', 'tail']
    if mode != 'fp32':
        assert p.convs['out_block.conv1'].cout in (cout, 16)             # padded to 16 as before (or folded, unpadded)


def test_more_than_127_classes_are_refused(monkeypatch):
    plan = _install(monkeypatch, [])
    sd = oinit.init_state_dict('vnet', 1, 128, 0)
    with pytest.raises(RuntimeError, match='int8'):
        plan.NetPlan(sd, mode='fp16', device='cpu')


@pytest.mark.parametrize('mode', ['bf16', 'fp32'])
def test_training_a_wide_net_raises(monkeypatch, mode):
    plan = _install(monkeypatch, [])
    p = plan.NetPlan(oinit.init_state_dict('vnet', 1, 17, 0), mode=mode, device='cpu')
    with pytest.raises(RuntimeError, match='training supports up to 16 classes'):
        p.plan(1, 16, 16, 16, train=True)
