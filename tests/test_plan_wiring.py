"""CPU check of the HOST WIRING of the whole-network kernel plan (segmentation3d/_b200/plan.py) against the oracle.

Every C-ABI entry point the forward plan issues is replaced by a torch emulation of its documented semantics
(include/seg3d_b200.h: NDHWC pitches and channel offsets, packed weight layouts of every convolution flavour, GroupNorm
sums, in-place concat, residual / ReLU flags, the folded narrow-output layout and its fused GroupNorm input, the split
hi/lo format of the strict mode), "device" tensors are CPU tensors and the plan's CUDA-only guard is stubbed.  What runs
for real is the plan: buffer allocation, views and offsets, weight packing, the order of ~60 calls per forward, for VNet and
VBNet in every execution mode.  A host-side regression in the plan then fails the CPU gate; the kernels themselves are
pinned by the `-m gpu` tests."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import init as oinit
from oracle import net as onet


class _P(object):
    def __init__(self, t, off):
        self.t, self.off = t, off

    def flat(self):
        return self.t.reshape(-1)[self.off:]


def _rows(p, n_rows, ld, C):
    """[n_rows, C] view of the flat buffer behind pointer p (element offset p.off, pitch ld)"""
    flat = p.t.reshape(-1)
    assert p.off + (n_rows - 1) * ld + C <= flat.numel(), 'kernel argument runs past its buffer'
    return torch.as_strided(flat, (n_rows, C), (ld, 1), p.off)


def _stats(y):
    return y.double().flatten(1).sum(1), (y.double() ** 2).flatten(1).sum(1)


def _stat_rows(stats, N):
    """[N, 2] view of the double sums behind pointer `stats` (element offset honoured: a sub-batch starts at sample b0)"""
    return stats.t.reshape(-1)[stats.off:stats.off + 2 * N].view(N, 2)


def _mean_rstd(stats, cnt, eps, N):
    rows = _stat_rows(stats, N)
    mean = (rows[:, 0] / cnt).view(N, 1, 1)
    var = (rows[:, 1] / cnt).view(N, 1, 1) - mean * mean
    return mean, 1.0 / torch.sqrt(var + eps)


def emulate_gather_pack(table, block_map, n_blocks, stream):
    """seg3d_gather_pack per include/seg3d_b200.h on HOST memory: the table holds raw addresses (CPU tensors here)"""
    import ctypes
    from segmentation3d._b200 import lib
    raw = bytes(table.t.reshape(-1)[table.off:].numpy().tobytes())
    bm = block_map.flat()[:2 * n_blocks].view(-1, 2)
    n_entries = int(bm[:, 0].max()) + 1
    entries = (lib.PackEntry * n_entries).from_buffer_copy(raw[:n_entries * ctypes.sizeof(lib.PackEntry)])
    for k, e in enumerate(entries):
        chunks = bm[bm[:, 0] == k][:, 1].tolist()
        n_e = int(np.prod(list(e.size)))
        assert chunks == list(range((n_e + lib.PACK_CHUNK - 1) // lib.PACK_CHUNK)), 'every chunk of every entry exactly once'
        size, limit = list(e.size), list(e.limit)
        idx = np.indices(size).reshape(5, -1)
        n = idx.shape[1]
        so = e.src_base + sum(idx[d] * e.src_stride[d] for d in range(5))
        do = e.dst_base + sum(idx[d] * e.dst_stride[d] for d in range(5))
        inside = np.ones(n, bool)
        for d in range(5):
            inside &= idx[d] < limit[d]
        assert so[inside].min() >= 0 and do.min() >= 0 and len(np.unique(do)) == n
        src = np.ctypeslib.as_array((ctypes.c_float * int(so[inside].max() + 1)).from_address(e.src))
        vals = np.where(inside, src[np.where(inside, so, 0)], np.float32(0)).astype(np.float32)
        if e.kind != lib.PACK_PLAIN:
            hi = vals.astype(np.float16).astype(np.float32)
            vals = hi if e.kind == lib.PACK_SPLIT_HI else vals - hi
        nd = int(do.max() + 1)
        if e.dtype == lib.F32:
            np.ctypeslib.as_array((ctypes.c_float * nd).from_address(e.dst))[do] = vals
        else:
            bits = torch.from_numpy(vals).to(lib.TORCH_DTYPE[e.dtype]).view(torch.int16).numpy()
            np.ctypeslib.as_array((ctypes.c_int16 * nd).from_address(e.dst))[do] = bits
    return 0


def _install(monkeypatch, calls):
    from segmentation3d._b200 import lib, plan

    def ptr(t, off=0):
        return None if t is None else _P(t, off)

    def _conv(mode, simt, xs, w, bias, Cin, Cout):
        wp = w.t.float().reshape(-1)
        k = {lib.CONV_K3: 3, lib.CONV_K2S2: 2, lib.CONV_T2S2: 2, lib.CONV_K1: 1}[mode]
        b = None if bias is None else bias.t.float()[:Cout]
        if mode == lib.CONV_T2S2:
            wt = wp[:Cin * 8 * Cout].view(Cin, 2, 2, 2, Cout) if simt else wp[:8 * Cout * Cin].view(2, 2, 2, Cout, Cin).permute(4, 0, 1, 2, 3)
            return F.conv_transpose3d(xs, wt.permute(0, 4, 1, 2, 3), b, stride=2)
        n = k ** 3 * Cin * Cout
        wt = wp[:n].view(k, k, k, Cin, Cout).permute(4, 3, 0, 1, 2) if simt else wp[:n].view(k, k, k, Cout, Cin).permute(3, 4, 0, 1, 2)
        return F.conv3d(xs, wt, b, stride=2 if mode == lib.CONV_K2S2 else 1, padding=1 if mode == lib.CONV_K3 else 0)

    def _store(r, y, y_ld, C, stats, N):
        if stats is not None:
            s0, s1 = _stats(r)
            st = _stat_rows(stats, N)
            st[:N, 0] += s0
            st[:N, 1] += s1
        rn = r.permute(0, 2, 3, 4, 1).reshape(-1, r.shape[1])
        dst = _rows(y, rn.shape[0], y_ld, C)
        dst.copy_(rn[:, :C].to(dst.dtype))

    def conv3d_fwd(mode, dtype, impl, x, x_ld, Cin, w, bias, y, y_ld, Cout, N, D, H, W, stats, stream):
        out_f32 = bool(dtype & lib.OUT_F32)
        xs = _rows(x, N * D * H * W, x_ld, Cin).float().view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        simt = impl == lib.IMPL_SIMT or (impl == lib.IMPL_AUTO and Cin == 1)
        r = _conv(mode, simt, xs, w, bias, Cin, Cout)
        if out_f32:
            assert y.t.dtype == torch.float32
        _store(r, y, y_ld, min(Cout, y_ld) if out_f32 else Cout, stats, N)
        calls.append('conv')
        return 0

    def cin1_fwd(dtype, epi, xpad, x_pitch, w, bias, y, y_ld, N, D, H, W, stats, gamma, beta, eps, stream):
        # row-padded single-channel input: x index i at column i + CIN1_LEFT, every other column zero
        assert x_pitch == W + lib.CIN1_PAD and W % 8 == 0
        rows = _rows(xpad, N * D * H, x_pitch, x_pitch).float()
        assert float(rows[:, :lib.CIN1_LEFT].abs().max()) == 0 and float(rows[:, lib.CIN1_LEFT + W:].abs().max()) == 0
        xs = rows[:, lib.CIN1_LEFT:lib.CIN1_LEFT + W].reshape(N, 1, D, H, W)
        # the kernel rounds the fp32 weights of the SIMT layout to the storage type (csrc/conv_tc_cin1t.cu); emulated for fp16,
        # the inference storage type (the bf16 backward wiring tests compare against fp32 autograd and keep the fp32 weights)
        if dtype == lib.F16:
            w = _P(w.t.float().half().float(), 0)
        r = _conv(lib.CONV_K3, True, xs, w, bias, 1, 16)
        if epi in (0, 1):
            s0, s1 = _stats(r)
            st = _stat_rows(stats, N)
            st[:N, 0] += s0
            st[:N, 1] += s1
        if epi == 1:
            assert y is None
            calls.append('conv_stats')
            return 0
        rn = r.permute(0, 2, 3, 4, 1).reshape(N, D * H * W, 16)
        if epi == 2:
            mean, rstd = _mean_rstd(stats, float(D * H * W * 16), eps, N)
            rn = F.relu(((rn.double() - mean) * rstd).float() * gamma.t.view(1, 1, 16) + beta.t.view(1, 1, 16))
        dst = _rows(y, N * D * H * W, y_ld, 16)
        dst.copy_(rn.reshape(-1, 16).to(dst.dtype))
        calls.append('conv')
        return 0

    def narrow_np(Cout):
        return (9 * Cout + 15) // 16 * 16

    def _narrow(xs, w, bias, Cin, Cout):
        NP = narrow_np(Cout)
        wf = w.t.float().view(3, NP, Cin)[:, :9 * Cout].view(3, 3, 3, Cout, Cin)            # [kd][kh][kw][co][ci]
        return F.conv3d(xs, wf.permute(3, 4, 0, 1, 2), bias.t.float()[:Cout], padding=1)

    def narrow_fwd(dtype, x, x_ld, Cin, w, bias, y, Cout, N, D, H, W, stats, stream):
        xs = _rows(x, N * D * H * W, x_ld, Cin).float().view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        _store(_narrow(xs, w, bias, Cin, Cout), y, Cout, Cout, stats, N)
        calls.append('narrow')
        return 0

    def gnin_fwd(dtype, x, x_ld, Cin, gn_ch, gn_stats, gamma, beta, eps, w, bias, y, y_ld, Cout, N, D, H, W, stats, stream):
        # the first gn_ch input channels are raw: relu(GroupNorm(1, gn_ch)) of them, rounded to the storage type, on load
        nvox = D * H * W
        xr = _rows(x, N * nvox, x_ld, Cin).float().view(N, nvox, Cin).clone()
        mean, rstd = _mean_rstd(gn_stats, float(nvox * gn_ch), eps, N)
        z = ((xr[..., :gn_ch].double() - mean) * rstd).float() * gamma.t[:gn_ch].view(1, 1, gn_ch) + beta.t[:gn_ch].view(1, 1, gn_ch)
        xr[..., :gn_ch] = F.relu(z).to(x.t.dtype).float()
        xs = xr.view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        _store(_conv(lib.CONV_K3, False, xs, w, bias, Cin, Cout), y, y_ld, Cout, stats, N)
        calls.append('conv_gnin')
        return 0

    def narrow_gn2_fwd(dtype, raw, raw_ld, res, res_ld, Cin, gn_stats, gamma, beta, eps, rg_ch, rg_stats, rg_gamma, rg_beta,
                       w, bias, y, Cout, N, D, H, W, stats, stream):
        nvox = D * H * W
        rr = _rows(res, N * nvox, res_ld, Cin).float().view(N, nvox, Cin).clone()
        mean, rstd = _mean_rstd(rg_stats, float(nvox * rg_ch), eps, N)
        z = ((rr[..., :rg_ch].double() - mean) * rstd).float() * rg_gamma.t[:rg_ch].view(1, 1, rg_ch) + rg_beta.t[:rg_ch].view(1, 1, rg_ch)
        rr[..., :rg_ch] = F.relu(z).to(res.t.dtype).float()
        resolved = _P(rr.reshape(-1).to(res.t.dtype), 0)
        rc = narrow_gn_fwd(dtype, raw, raw_ld, resolved, Cin, Cin, gn_stats, gamma, beta, eps, w, bias, y, Cout, N, D, H, W, stats, stream)
        calls[-1] = 'narrow_gn2'
        return rc

    def narrow_split_fwd(x, x_ld, Cin, w, bias, y, Cout, N, D, H, W, stats, stream):
        rows = N * D * H * W
        assert Cin == 32 and x_ld >= 64
        xs = (_rows(x, rows, x_ld, Cin).float() + _rows(_P(x.t, x.off + Cin), rows, x_ld, Cin).float())
        xs = xs.view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        wq = w.t.float().view(3, narrow_np(Cout), 2 * Cin)                                # rows [whi(Cin) | wlo(Cin)]
        wsum = _P((wq[..., :Cin] + wq[..., Cin:]).contiguous(), 0)
        _store(_narrow(xs, wsum, bias, Cin, Cout), y, Cout, Cout, stats, N)
        calls.append('narrow')
        return 0

    def narrow_gn_fwd(dtype, raw, raw_ld, res, res_ld, Cin, gn_stats, gamma, beta, eps, w, bias, y, Cout, N, D, H, W, stats, stream):
        nvox = D * H * W
        r = _rows(raw, N * nvox, raw_ld, Cin).float().view(N, nvox, Cin)
        mean, rstd = _mean_rstd(gn_stats, float(nvox * Cin), eps, N)
        z = ((r.double() - mean) * rstd).float() * gamma.t.view(1, 1, Cin) + beta.t.view(1, 1, Cin)
        z = F.relu(z + _rows(res, N * nvox, res_ld, Cin).float().view(N, nvox, Cin)).to(raw.t.dtype).float()   # stored type in smem
        xs = z.view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        _store(_narrow(xs, w, bias, Cin, Cout), y, Cout, Cout, stats, N)
        calls.append('narrow_gn')
        return 0

    def gn_apply(dtype, y, y_ld, C, stats, gamma, beta, eps, res, res_ld, out, out_ld, relu, N, nvox, stream):
        ys = _rows(y, N * nvox, y_ld, C).float().view(N, nvox, C)
        mean, rstd = _mean_rstd(stats, float(nvox * C), eps, N)
        z = ((ys.double() - mean) * rstd).float() * gamma.t.view(1, 1, C) + beta.t.view(1, 1, C)
        if res is not None:
            z = z + _rows(res, N * nvox, res_ld, C).float().view(N, nvox, C)
        if relu:
            z = F.relu(z)
        dst = _rows(out, N * nvox, out_ld, C)
        dst.copy_(z.reshape(-1, C).to(dst.dtype))
        calls.append('gn')
        return 0

    def split_fwd(mode, x, x_ld, lo_off, Cin, w, bias, y, y_ld, Cout, N, D, H, W, stats, stream):
        rows = N * D * H * W
        xs = (_rows(x, rows, x_ld, Cin).float() + _rows(_P(x.t, x.off + lo_off), rows, x_ld, Cin).float())
        xs = xs.view(N, D, H, W, Cin).permute(0, 4, 1, 2, 3)
        wq = w.t.float()                                                              # [..][Cout][whi(Cin) | wlo(Cin)]
        wsum = _P((wq[..., :Cin] + wq[..., Cin:]).contiguous(), 0)
        _store(_conv(mode, False, xs, wsum, bias, Cin, Cout), y, y_ld, Cout, stats, N)
        calls.append('split_conv')
        return 0

    def gn_apply_split(y, y_ld, C, stats, gamma, beta, eps, res, res_ld, res_lo, out, out_ld, out_lo, relu, N, nvox, stream):
        ys = _rows(y, N * nvox, y_ld, C).float().view(N, nvox, C)
        mean, rstd = _mean_rstd(stats, float(nvox * C), eps, N)
        z = ((ys.double() - mean) * rstd).float() * gamma.t.view(1, 1, C) + beta.t.view(1, 1, C)
        if res is not None:
            z = z + (_rows(res, N * nvox, res_ld, C).float() + _rows(_P(res.t, res.off + res_lo), N * nvox, res_ld, C).float()).view(N, nvox, C)
        if relu:
            z = F.relu(z)
        z = z.reshape(-1, C)
        hi = z.half()
        _rows(out, N * nvox, out_ld, C).copy_(hi)
        _rows(_P(out.t, out.off + out_lo), N * nvox, out_ld, C).copy_((z - hi.float()).half())
        calls.append('gn_split')
        return 0

    def _tail(y1, ld, C, stats1, g1, b1, w2, bias2, eps, N, nvox):
        ys = _rows(y1, N * nvox, ld, C).float().view(N, nvox, C)
        mean, rstd = _mean_rstd(stats1, float(nvox * C), eps, N)
        a = F.relu(((ys.double() - mean) * rstd).float() * g1.t.view(1, 1, C) + b1.t.view(1, 1, C))
        return a @ w2.t.view(C, C).t() + bias2.t.view(1, 1, C)

    def tail_stats(dtype, y1, ld, C, stats1, g1, b1, w2, bias2, eps, stats2, N, nvox, stream):
        z = _tail(y1, ld, C, stats1, g1, b1, w2, bias2, eps, N, nvox)
        rows = _stat_rows(stats2, N)
        rows[:, 0] += z.double().flatten(1).sum(1)
        rows[:, 1] += (z.double() ** 2).flatten(1).sum(1)
        calls.append('tail_stats')
        return 0

    def tail_probs(dtype, y1, ld, C, stats1, g1, b1, w2, bias2, stats2, g2, b2, eps, probs, N, nvox, stream):
        z = _tail(y1, ld, C, stats1, g1, b1, w2, bias2, eps, N, nvox)
        mean, rstd = _mean_rstd(stats2, float(nvox * C), eps, N)
        z = ((z.double() - mean) * rstd).float() * g2.t.view(1, 1, C) + b2.t.view(1, 1, C)
        dst = probs.t.reshape(-1)[probs.off:probs.off + N * C * nvox]
        dst.copy_(F.softmax(z, 2).permute(0, 2, 1).reshape(-1))
        calls.append('tail_probs')
        return 0

    table = {'seg3d_conv3d_fwd': conv3d_fwd, 'seg3d_conv3d_cin1_fwd': cin1_fwd, 'seg3d_conv3d_k3_narrow_split_fwd': narrow_split_fwd,
             'seg3d_conv3d_k3_gnin_fwd': gnin_fwd, 'seg3d_conv3d_k3_narrow_gn2_fwd': narrow_gn2_fwd,
             'seg3d_conv3d_k3_narrow_fwd': narrow_fwd, 'seg3d_conv3d_k3_narrow_gn_fwd': narrow_gn_fwd,
             'seg3d_gn_apply': gn_apply, 'seg3d_conv3d_split_fwd': split_fwd, 'seg3d_gn_apply_split': gn_apply_split,
             'seg3d_outblock_tail_stats': tail_stats, 'seg3d_outblock_tail_probs': tail_probs,
             'seg3d_gather_pack': emulate_gather_pack}
    monkeypatch.setattr(lib, 'ptr', ptr)
    monkeypatch.setattr(lib, 'call', lambda name, *a: table[name](*a))
    monkeypatch.setattr(lib, 'stream_ptr', lambda: 0)
    monkeypatch.setattr(plan, '_require_cuda', lambda device, message: None)         # the test stubs the guard, the package never does
    return plan


@pytest.mark.parametrize('arch,cout', [('vnet', 2), ('vbnet', 5)])
@pytest.mark.parametrize('mode,tol', [('fp32', 2e-5), ('fp16', 2e-2), ('bf16', 1.5e-1), ('fp32x', 1e-4)])
def test_plan_issues_the_reference_network(monkeypatch, arch, cout, mode, tol):
    calls = []
    plan = _install(monkeypatch, calls)
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 7)
    x = torch.randn((2, 1, 16, 32, 16), generator=torch.Generator().manual_seed(3))
    ref = onet.forward(sd, x)
    p = plan.NetPlan(sd, mode=mode, device='cpu')
    got = p.forward(x).clone()
    assert got.shape == ref.shape and got.dtype == torch.float32
    err = float((got - ref).abs().max())
    assert err <= tol, (arch, mode, err)
    assert float((got.sum(1) - 1).abs().max()) <= 1e-5
    n_convs = sum(1 for k, v in sd.items() if k.endswith('.weight') and v.dim() == 5) - 1          # out_block.conv2 lives in the tail
    assert sum(c in ('conv', 'conv_gnin', 'narrow', 'narrow_gn', 'narrow_gn2', 'split_conv') for c in calls) == n_convs
    if mode in ('fp16', 'bf16'):
        assert 'conv_stats' in calls                                                  # input block: statistics pass + fused GroupNorm/ReLU pass
        # fused last GroupNorm + narrow-output conv is the default; up_32.up_gn is applied on load by both of its readers
        assert 'conv_gnin' in calls and 'narrow_gn2' in calls
    if mode == 'fp32x':
        assert 'split_conv' in calls and 'gn_split' in calls
    # a second forward through the cached plan, and after an in-place weight refresh, stays correct
    sd2 = {k: (v * 1.01 if k.endswith('conv.weight') else v) for k, v in sd.items()}
    p.refresh(sd2)
    err = float((p.forward(x) - onet.forward(sd2, x)).abs().max())
    assert err <= tol, (arch, mode, 'refresh', err)


@pytest.mark.parametrize('arch,cout,mode', [('vnet', 2, 'fp16'), ('vbnet', 5, 'fp32x'), ('vnet', 3, 'fp32')])
def test_sub_batched_schedule_is_the_same_network(monkeypatch, arch, cout, mode):
    """plan.py::_schedule: the level 0 / 1 runs issued in sub-batches (pointer offsets per sample, the raw scratch re-used in
    place) give the probabilities of the whole-batch schedule, also for a ragged last sub-batch"""
    calls = []
    plan = _install(monkeypatch, calls)
    monkeypatch.delenv('SEG3D_MODE', raising=False)
    sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 9)
    x = torch.randn((5, 1, 16, 16, 32), generator=torch.Generator().manual_seed(4))
    monkeypatch.setenv('SEG3D_SUBBATCH_MB', '0')
    p0 = plan.NetPlan(sd, mode=mode, device='cpu')
    whole = p0.forward(x).clone()
    n0 = len(calls)
    assert p0.launches_per_forward == n0
    per_sample_mb = 16 * 16 * 32 * 32 * (4 if mode == 'fp32' else (4 if mode == 'fp32x' else 2)) / 1e6
    monkeypatch.setenv('SEG3D_SUBBATCH_MB', str(2.5 * per_sample_mb))        # sub-batches of 2, 2, 1
    del calls[:]
    p1 = plan.NetPlan(sd, mode=mode, device='cpu')
    ws, ops = p1.plan(5, 16, 16, 32)
    assert [sb for _, _, sb in ws['schedule']] == [2, 5, 2] and sum(i1 - i0 for i0, i1, _ in ws['schedule']) == len(ops)
    sub = p1.forward(x).clone()
    # (the CPU emulation's convolutions sum in a batch-size dependent order, and a half-precision store can flip on that)
    assert float((whole - sub).abs().max()) <= (2e-3 if mode == 'fp16' else 1e-5)
    assert len(calls) == p1.launches_per_forward > n0
    assert float((sub - onet.forward(sd, x)).abs().max()) <= (2e-5 if mode == 'fp32' else (1e-4 if mode == 'fp32x' else 2e-2))


def test_plan_without_the_fused_tail_and_with_batches(monkeypatch):
    calls = []
    plan = _install(monkeypatch, calls)
    sd = oinit.randomize_affine(oinit.init_state_dict('vnet', 1, 2, 1), 2)
    g = torch.Generator().manual_seed(5)
    x = torch.randn((3, 1, 16, 16, 32), generator=g)
    ref = onet.forward(sd, x)
    for env in ({'SEG3D_FUSE_TAIL': '0'}, {'SEG3D_NARROW': '0'}, {'SEG3D_TAIL_F32': '0'}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        del calls[:]
        got = plan.NetPlan(sd, mode='fp16', device='cpu').forward(x)
        assert float((got - ref).abs().max()) <= 2e-2, env
        assert 'narrow_gn' not in calls
        for k in env:
            monkeypatch.delenv(k)
    # GroupNorm is per sample: a batch equals its items run one by one
    p = plan.NetPlan(sd, mode='fp32', device='cpu')
    whole = p.forward(x).clone()
    for i in range(3):
        assert float((p.forward(x[i:i + 1]) - whole[i:i + 1]).abs().max()) <= 1e-5


@pytest.mark.parametrize('arch,cout,mode,tol', [('vnet', 2, 'fp16', 2e-2), ('vbnet', 5, 'fp32x', 1e-4), ('vnet', 3, 'fp32', 2e-5)])
def test_bound_plan_repacks_changed_weights_with_one_launch(monkeypatch, arch, cout, mode, tol):
    """network/_graph.py binds the plan to the live parameters: after an in-place weight change the next forward re-packs
    every layout (tensor-core, folded narrow-output, split hi/lo, SIMT, biases, GroupNorm affines) through the gather table"""
    import importlib
    calls = []
    plan = _install(monkeypatch, calls)
    real = plan.lib.call
    seen = []
    monkeypatch.setattr(plan.lib, 'call', lambda name, *a: (seen.append(name), real(name, *a))[1])
    mod = importlib.import_module('segmentation3d.network.' + arch)
    net = mod.SegmentationNet(1, cout)
    net.load_state_dict(oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 5))
    net.b200_mode = mode
    net.eval()
    x = torch.randn((1, 1, 16, 16, 32), generator=torch.Generator().manual_seed(8))
    with torch.no_grad():
        assert float((net(x) - onet.forward(net.state_dict(), x)).abs().max()) <= tol
        assert 'seg3d_gather_pack' not in seen
        g = torch.Generator().manual_seed(1)
        for p in net.parameters():
            p.mul_(1.0 + 0.05 * torch.randn(p.shape, generator=g)).add_(0.01 * torch.randn(p.shape, generator=g))
        err = float((net(x) - onet.forward(net.state_dict(), x)).abs().max())
    assert seen.count('seg3d_gather_pack') == 1
    assert err <= tol, (arch, mode, err)
