"""Kernel calls behind the STANDALONE network modules (segmentation3d/network/module/*.py).

`SegmentationNet` runs a whole-network plan (plan.py: workspaces allocated once, concat in place, fused tail).  The
reference also exposes its building blocks as importable nn.Modules (network/module/conv_gn_relu3.py, residual_block3.py,
vnet_inblock.py, vnet_downblock.py, vnet_upblock.py, vnet_outblock.py); the classes in network/module keep those
constructors and state-dict keys and run their forward through the same C-ABI entry points, one conv -> GroupNorm unit at
a time: NCDHW fp32 in and out like the reference modules, NDHWC in the mode's storage type in between.  Inference only
(the training path differentiates the whole-network plan); no torch arithmetic, no CPU path.

STATUS: written at the end of round 1 after the GPU budget was spent - the call patterns are those of plan.py, but these
wrappers have not run on a GPU yet; their parity tests (tests/test_gpu_blocks.py) are skipped unless SEG3D_TEST_UNVERIFIED=1.
"""
import os

import torch

from . import lib
from .plan import DEFAULT_TC_MODES, GN_EPS, MODES, WIDE_MAX_CLASSES, _Conv


def block_mode(module):
    mode = getattr(module, 'b200_mode', None) or os.environ.get('SEG3D_MODE', 'fp16')
    if mode not in ('fp32', 'fp16', 'bf16'):
        raise RuntimeError("standalone network modules run in 'fp32', 'fp16' or 'bf16' (got %r); 'fp32x' is a whole-network mode" % mode)
    return mode, MODES[mode]


def check_input(x, channels):
    if not (torch.is_tensor(x) and x.is_cuda):
        raise RuntimeError('segmentation3d (B200 build) has no CPU path: pass a CUDA tensor')
    if x.dim() != 5 or x.shape[1] != channels:
        raise ValueError('expected a [B, %d, D, H, W] tensor, got %s' % (channels, tuple(x.shape)))
    if torch.is_grad_enabled() and x.requires_grad:
        raise RuntimeError('standalone network modules are inference-only: train through SegmentationNet')


def to_ndhwc(x, dt):
    """[B,C,D,H,W] float32 -> [B,D,H,W,C] in the storage type of `dt`."""
    return x.detach().permute(0, 2, 3, 4, 1).contiguous().to(lib.TORCH_DTYPE[dt])


def to_ncdhw(y):
    return y.permute(0, 4, 1, 2, 3).float().contiguous()


def packed_conv(holder, conv_mode, dt, pad_cout=0):
    """weights of a Conv3dParams / ConvTranspose3dParams holder packed for the kernels (plan._Conv), cached on the holder
    and re-packed in place when the parameters change."""
    w, b = holder.weight, holder.bias
    key = (conv_mode, dt, str(w.device), w._version, w.data_ptr(), None if b is None else (b._version, b.data_ptr()))
    cache = holder.__dict__.setdefault('_b200_packed', {})
    ent = cache.get((conv_mode, dt))
    sd = {'c.weight': w.detach()}
    if b is not None:
        sd['c.bias'] = b.detach()
    else:
        sd['c.bias'] = torch.zeros((w.shape[1] if conv_mode == lib.CONV_T2S2 else w.shape[0],), device=w.device)
    if ent is None or ent[0][2] != key[2]:
        conv = _Conv(sd, 'c', conv_mode, dt, w.device, DEFAULT_TC_MODES, pad_cout=pad_cout)
        cache[(conv_mode, dt)] = (key, conv)
        return conv
    if ent[0] != key:
        ent[1].load(sd)
        cache[(conv_mode, dt)] = (key, ent[1])
    return ent[1]


def out_dims(conv_mode, D, H, W):
    if conv_mode == lib.CONV_K2S2:
        if D % 2 or H % 2 or W % 2:
            raise ValueError('stride-2 convolution needs even spatial dims')
        return D // 2, H // 2, W // 2
    if conv_mode == lib.CONV_T2S2:
        return 2 * D, 2 * H, 2 * W
    return D, H, W


def conv_raw(x_nd, holder, conv_mode, dt, pad_cout=0):
    """raw convolution + bias and its per-sample GroupNorm sums: ([B,Do,Ho,Wo,Cout'] storage type, double [B,2], conv)."""
    B, D, H, W, cin = x_nd.shape
    conv = packed_conv(holder, conv_mode, dt, pad_cout)
    if conv.cin != cin:
        raise ValueError('convolution expects %d input channels, got %d' % (conv.cin, cin))
    Do, Ho, Wo = out_dims(conv_mode, D, H, W)
    raw = torch.empty((B, Do, Ho, Wo, conv.cout), dtype=lib.TORCH_DTYPE[dt], device=x_nd.device)
    stats = torch.zeros((B, 2), dtype=torch.float64, device=x_nd.device)
    with torch.cuda.device(x_nd.device):
        lib.call('seg3d_conv3d_fwd', conv.mode, dt, conv.call_impl, lib.ptr(x_nd), cin, cin, lib.ptr(conv.w), lib.ptr(conv.bias),
                 lib.ptr(raw), conv.cout, conv.cout, B, D, H, W, lib.ptr(stats), lib.stream_ptr())
    return raw, stats, conv


def gn_apply(raw, stats, gn_holder, dt, relu, res=None, out=None, out_off=0):
    """out[..., out_off:out_off+C] = [relu](GroupNorm(raw) [+ res]); `out` defaults to a fresh dense tensor."""
    B, D, H, W, C = raw.shape
    if out is None:
        out, out_off = torch.empty_like(raw), 0
    gamma = gn_holder.weight.detach().float().contiguous()
    beta = gn_holder.bias.detach().float().contiguous()
    with torch.cuda.device(raw.device):
        lib.call('seg3d_gn_apply', dt, lib.ptr(raw), C, C, lib.ptr(stats), lib.ptr(gamma), lib.ptr(beta), GN_EPS,
                 lib.ptr(res) if res is not None else None, res.shape[-1] if res is not None else 0,
                 lib.ptr(out, out_off), out.shape[-1], 1 if relu else 0, B, D * H * W, lib.stream_ptr())
    return out


def conv_gn(x_nd, conv_holder, gn_holder, conv_mode, dt, relu, res=None, out=None, out_off=0):
    raw, stats, _ = conv_raw(x_nd, conv_holder, conv_mode, dt)
    return gn_apply(raw, stats, gn_holder, dt, relu, res, out, out_off)


def output_tail(x_nd, conv1, gn1, conv2, gn2, dt):
    """vnet_outblock.py:20-24: conv1 -> GN1 -> ReLU -> 1x1x1 conv2 -> GN2 -> softmax; fp32 [B,C,D,H,W] probabilities."""
    B, D, H, W, cin = x_nd.shape
    nc = conv1.weight.shape[0]
    if nc > WIDE_MAX_CLASSES:
        raise RuntimeError('seg3d_b200: at most %d output classes are supported: the label mask is int8' % WIDE_MAX_CLASSES)
    s2 = torch.zeros((B, 2), dtype=torch.float64, device=x_nd.device)
    g1w, g1b = gn1.weight.detach().float().contiguous(), gn1.bias.detach().float().contiguous()
    g2w, g2b = gn2.weight.detach().float().contiguous(), gn2.bias.detach().float().contiguous()
    w2 = conv2.weight.detach().float().reshape(nc, nc).contiguous()
    b2 = conv2.bias.detach().float().contiguous()
    probs = torch.empty((B, nc, D, H, W), dtype=torch.float32, device=x_nd.device)
    nvox = D * H * W
    if nc > 16:
        # the whole-network plan's wide path: conv1 zero-padded to Cp channels, its raw result in fp32 rows of pitch Cp, then
        # the tensor-core tail (csrc/tail_wide.cu)
        cp = (nc + 15) // 16 * 16
        c1 = packed_conv(conv1, lib.CONV_K3, dt, pad_cout=cp)
        if c1.cin != cin:
            raise ValueError('convolution expects %d input channels, got %d' % (c1.cin, cin))
        raw = torch.empty((B, D, H, W, cp), dtype=torch.float32, device=x_nd.device)
        s1 = torch.zeros((B, 2), dtype=torch.float64, device=x_nd.device)
        with torch.cuda.device(x_nd.device):
            lib.call('seg3d_conv3d_fwd', c1.mode, dt if dt == lib.F32 else dt | lib.OUT_F32, c1.call_impl, lib.ptr(x_nd), cin, cin,
                     lib.ptr(c1.w), lib.ptr(c1.bias), lib.ptr(raw), cp, c1.cout, B, D, H, W, lib.ptr(s1), lib.stream_ptr())
            for ps in (0, 1):
                lib.call('seg3d_outblock_tail_wide', ps, lib.ptr(raw), cp, nc, lib.ptr(s1), lib.ptr(g1w), lib.ptr(g1b), lib.ptr(w2),
                         lib.ptr(b2), GN_EPS, lib.ptr(s2), lib.ptr(g2w), lib.ptr(g2b), lib.ptr(probs), B, nvox, lib.stream_ptr())
        return probs
    raw, s1, c1 = conv_raw(x_nd, conv1, lib.CONV_K3, dt, pad_cout=16)
    with torch.cuda.device(x_nd.device):
        lib.call('seg3d_outblock_tail_stats', dt, lib.ptr(raw), c1.cout, nc, lib.ptr(s1), lib.ptr(g1w), lib.ptr(g1b), lib.ptr(w2),
                 lib.ptr(b2), GN_EPS, lib.ptr(s2), B, nvox, lib.stream_ptr())
        lib.call('seg3d_outblock_tail_probs', dt, lib.ptr(raw), c1.cout, nc, lib.ptr(s1), lib.ptr(g1w), lib.ptr(g1b), lib.ptr(w2),
                 lib.ptr(b2), lib.ptr(s2), lib.ptr(g2w), lib.ptr(g2b), GN_EPS, lib.ptr(probs), B, nvox, lib.stream_ptr())
    return probs
