"""Kernel calls behind the STANDALONE network modules (segmentation3d/network/module/*.py).

`SegmentationNet` runs a whole-network plan (plan.py: workspaces allocated once, concat in place, fused tail).  The
reference also exposes its building blocks as importable nn.Modules (network/module/conv_gn_relu3.py, residual_block3.py,
vnet_inblock.py, vnet_downblock.py, vnet_upblock.py, vnet_outblock.py); the classes in network/module keep those
constructors and state-dict keys and run their forward through the same C-ABI entry points, one conv -> GroupNorm unit at
a time: NCDHW fp32 in and out like the reference modules, NDHWC in the mode's storage type in between.  No torch
arithmetic, no CPU path.

Training: a module call is differentiable under the predicate of SegmentationNet.forward extended to the inputs (grad
mode on, and an input or a parameter requires grad).  It then runs in the training mode of the whole network ('fp16' ->
'bf16', 'bf16', 'fp32'), issues the same forward launches while a `_Tape` keeps every unit's input view, raw conv output,
GroupNorm sums and output, and returns a tensor with one autograd node (`_ModuleFunction`).  Its backward turns the
incoming NCDHW gradient into NDHWC (seg3d_grad_from_ncdhw), walks the units in reverse with the per-unit step of the
whole-network backward (autograd.unit_step), and sums each input's gradient contributions into NCDHW fp32
(seg3d_grad_to_ncdhw).  Otherwise (torch.no_grad(), or nothing requires grad) the launches are those of inference.
"""
import os

import torch

from . import lib
from .autograd import _k3_dgrad_weight, _same_weight, unit_step
from .plan import DEFAULT_TC_MODES, GN_EPS, MODES, WIDE_MAX_CLASSES, _Conv, _View

TRAIN_MAX_CLASSES = 16        # the out-block tail backward (seg3d_outblock_tail_bwd), as for the whole network
_TAPS = {lib.CONV_K3: 27, lib.CONV_K2S2: 8, lib.CONV_T2S2: 8, lib.CONV_K1: 1}
# the data gradient of each convolution flavour: the forward kernel of the paired mode on a transformed weight
_DGRAD = {lib.CONV_K3: (lib.CONV_K3, _k3_dgrad_weight), lib.CONV_K1: (lib.CONV_K1, _k3_dgrad_weight),
          lib.CONV_K2S2: (lib.CONV_T2S2, _same_weight), lib.CONV_T2S2: (lib.CONV_K2S2, _same_weight)}


def block_mode(module, train=False):
    """(mode, storage dtype) of a module call; a training call runs in the mode the whole network trains in
    (VShapedNet.resolve_mode(train=True)): 'fp16' (the default) -> 'bf16', 'bf16' and 'fp32' as given."""
    mode = getattr(module, 'b200_mode', None) or os.environ.get('SEG3D_MODE', 'fp16')
    if mode not in ('fp32', 'fp16', 'bf16'):
        raise RuntimeError("standalone network modules run in 'fp32', 'fp16' or 'bf16' (got %r); 'fp32x' is a whole-network mode" % mode)
    if train and mode != 'fp32':
        mode = 'bf16'
    return mode, MODES[mode]


def check_input(x, channels):
    if not (torch.is_tensor(x) and x.is_cuda):
        raise RuntimeError('segmentation3d (B200 build) has no CPU path: pass a CUDA tensor')
    if x.dim() != 5 or x.shape[1] != channels:
        raise ValueError('expected a [B, %d, D, H, W] tensor, got %s' % (channels, tuple(x.shape)))


def to_ndhwc(x, dt, tape=None, index=0):
    """[B,C,D,H,W] float32 -> [B,D,H,W,C] in the storage type of `dt` (a training call records it as module input `index`)."""
    y = x.detach().permute(0, 2, 3, 4, 1).contiguous().to(lib.TORCH_DTYPE[dt])
    if tape is not None:
        tape.input(index, _dense(y))
    return y


def to_ncdhw(y, tape=None):
    if tape is not None:
        tape.out = _dense(y)
    return y.permute(0, 4, 1, 2, 3).float().contiguous()


def _dense(t):
    return _View(t, 0, t.shape[-1], t.shape[-1])


def packed_conv(holder, conv_mode, dt, pad_cout=0, dgrad=False):
    """weights of a Conv3dParams / ConvTranspose3dParams holder packed for the kernels (plan._Conv), cached on the holder
    and re-packed in place when the parameters change.  dgrad=True: the weights of the data-gradient convolution (_DGRAD;
    zero-padded to the forward's `pad_cout` output channels when the forward ran padded)."""
    w, b = holder.weight, holder.bias
    key = (conv_mode, dt, str(w.device), w._version, w.data_ptr(), None if b is None else (b._version, b.data_ptr()))
    cache = holder.__dict__.setdefault('_b200_packed', {})
    ck = (conv_mode, dt, 'dgrad', pad_cout) if dgrad else (conv_mode, dt)
    ent = cache.get(ck)
    sd = {'c.weight': w.detach()}
    if b is not None:
        sd['c.bias'] = b.detach()
    else:
        sd['c.bias'] = torch.zeros((w.shape[1] if conv_mode == lib.CONV_T2S2 else w.shape[0],), device=w.device)
    if ent is None or ent[0][2] != key[2]:
        if dgrad:
            dmode, transform = _DGRAD[conv_mode]
            conv = _Conv(sd, 'c', dmode, dt, w.device, DEFAULT_TC_MODES, transform=transform, pad_dim0=pad_cout)
        else:
            conv = _Conv(sd, 'c', conv_mode, dt, w.device, DEFAULT_TC_MODES, pad_cout=pad_cout)
        cache[ck] = (key, conv)
        return conv
    if ent[0] != key:
        ent[1].load(sd)
        cache[ck] = (key, ent[1])
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


def conv_gn(x_nd, conv_holder, gn_holder, conv_mode, dt, relu, res=None, out=None, out_off=0, tape=None):
    raw, stats, conv = conv_raw(x_nd, conv_holder, conv_mode, dt)
    y = gn_apply(raw, stats, gn_holder, dt, relu, res, out, out_off)
    if tape is not None:
        tape.unit(x_nd, conv_holder, gn_holder, conv_mode, conv, raw, stats, y, out_off, relu, res)
    return y


def output_tail(x_nd, conv1, gn1, conv2, gn2, dt, tape=None):
    """vnet_outblock.py:20-24: conv1 -> GN1 -> ReLU -> 1x1x1 conv2 -> GN2 -> softmax; fp32 [B,C,D,H,W] probabilities."""
    B, D, H, W, cin = x_nd.shape
    nc = conv1.weight.shape[0]
    if nc > WIDE_MAX_CLASSES:
        raise RuntimeError('seg3d_b200: at most %d output classes are supported: the label mask is int8' % WIDE_MAX_CLASSES)
    if tape is not None and nc > TRAIN_MAX_CLASSES:
        raise RuntimeError('seg3d_b200: training supports up to %d classes (this block has %d); blocks with up to %d classes '
                           'run inference under torch.no_grad()' % (TRAIN_MAX_CLASSES, nc, WIDE_MAX_CLASSES))
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
    if tape is not None:
        tape.tail = dict(x=_dense(x_nd), conv1=conv1, gn1=gn1, conv2=conv2, gn2=gn2, c1=c1, raw=_dense(raw), s1=s1, s2=s2,
                         g1=(g1w, g1b), g2=(g2w, g2b), w2=w2, b2=b2, nc=nc)
    return probs


# ---- training ---------------------------------------------------------------------------------------------------------
def run_module(module, body, *inputs):
    """Forward of a standalone module: body(dt, tape, *inputs) issues the launches and returns the NCDHW fp32 result.
    Differentiable (one autograd node per call) when grad mode is on and an input or a parameter requires grad - the
    predicate of SegmentationNet.forward, extended to the inputs; otherwise exactly the inference launches."""
    params = list(module.parameters())
    if torch.is_grad_enabled() and (any(x.requires_grad for x in inputs) or any(p.requires_grad for p in params)):
        return _ModuleFunction.apply(module, body, len(inputs), *inputs, *params)
    _, dt = block_mode(module)
    return body(dt, None, *inputs)


class _ModuleFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, body, n_in, *args):
        inputs = args[:n_in]
        _, dt = block_mode(module, train=True)
        tape = _Tape(dt, inputs[0].device)
        with torch.no_grad():
            out = body(dt, tape, *inputs)
        ctx.tape, ctx.n_in, ctx.params = tape, n_in, args[n_in:]
        return out

    @staticmethod
    def backward(ctx, gout):
        need = ctx.needs_input_grad[3:3 + ctx.n_in]
        with torch.cuda.device(ctx.tape.device):
            din, dparam = ctx.tape.backward(gout, need)
        return (None, None, None) + tuple(din.get(i) for i in range(ctx.n_in)) + tuple(dparam.get(id(p)) for p in ctx.params)


class _Tape(object):
    """What a training forward of one module keeps for its backward: per conv -> GroupNorm unit its input view, raw conv
    output, GroupNorm sums, output view and residual view (plan._View windows of NDHWC buffers, as in the whole-network
    walk), the out-block tail's saved tensors, the NDHWC copies of the module's inputs and the output view."""

    def __init__(self, dt, device):
        self.dt, self.device = dt, device
        self.units, self.inputs, self.out, self.tail = [], {}, None, None

    def input(self, index, view):
        self.inputs[index] = view

    def unit(self, x_nd, conv_holder, gn_holder, conv_mode, conv, raw, stats, out, out_off, relu, res):
        self.units.append(dict(x=_dense(x_nd), conv=conv_holder, gn=gn_holder, mode=conv_mode, c=conv, raw=_dense(raw),
                               stats=stats, out=_View(out, out_off, out.shape[-1], conv.cout), relu=relu,
                               res=None if res is None else _dense(res), xd=x_nd.shape[1:4], od=raw.shape[1:4]))

    def backward(self, gout, need_input):
        dt, td, dev = self.dt, lib.TORCH_DTYPE[self.dt], self.device
        st = lib.stream_ptr
        # gradient targets: every unit's output and every module input that needs a gradient, keyed by (buffer, offset)
        targets = {(id(u['out'].buf), u['out'].off): u['out'] for u in self.units}
        for i, v in self.inputs.items():
            if need_input[i]:
                targets[(id(v.buf), v.off)] = v
        contrib = {}

        def inside(xv):
            return [(k, tv) for k, tv in targets.items() if k[0] == id(xv.buf) and xv.off <= k[1] and k[1] + tv.C <= xv.off + xv.C]

        def add_contrib(xv, gv):
            """register gradient view gv (same channel window as the consumer's input view xv) with every target inside xv"""
            for k, tv in inside(xv):
                contrib.setdefault(k, []).append(_View(gv.buf, gv.off + (k[1] - xv.off), gv.ld, tv.C))

        # parameter-gradient slots in kernel layouts: fp32 views of one zeroed buffer
        sizes = []
        for u in self.units:
            c = u['c']
            sizes += [_TAPS[u['mode']] * c.cin * c.cout, c.cout, c.cout, c.cout]
        t = self.tail
        if t is not None:
            nc, c1 = t['nc'], t['c1']
            sizes += [27 * c1.cin * c1.cout, c1.cout, nc, nc, nc * nc, nc, nc, nc]
        offs, total = [], 0
        for n in sizes:
            offs.append(total)
            total += (n + 3) // 4 * 4
        flat = torch.zeros((total,), dtype=torch.float32, device=dev)
        slots = [flat[o:o + n] for o, n in zip(offs, sizes)]
        sums = torch.zeros((len(self.units) + 2, gout.shape[0], 2), dtype=torch.float64, device=dev)
        gout = gout.contiguous().float()
        B = gout.shape[0]
        grads = {}

        def conv_grads(holder, mode, c, dw, db):
            if mode == lib.CONV_T2S2:          # [Cin][tap][Cout] -> [Cin][Cout][a][b][c]
                g = dw.view(c.cin, 2, 2, 2, c.cout).permute(0, 4, 1, 2, 3)
            else:                              # [tap][Cin][Cout] -> [Cout][Cin][a][b][c]
                k = {lib.CONV_K3: 3, lib.CONV_K2S2: 2, lib.CONV_K1: 1}[mode]
                g = dw.view(k, k, k, c.cin, c.cout)[..., :c.real_cout].permute(4, 3, 0, 1, 2)
            grads[id(holder.weight)] = g.contiguous()
            if holder.bias is not None:
                grads[id(holder.bias)] = db[:c.real_cout]

        def dgrad_of(holder, mode, c, x, od, pad_cout=0):
            """(dgrad convolution, gradient view, gy dims) when a target lies inside the unit's input x, else None"""
            if not inside(x):
                return None
            dcv = packed_conv(holder, mode, dt, pad_cout=pad_cout, dgrad=True)
            gd = torch.empty(tuple(x.buf.shape[:4]) + (dcv.cout,), dtype=td, device=dev)
            return dcv, _dense(gd), od

        # ---- where the module's output gradient enters --------------------------------------------------------------
        if t is not None:
            x, c1, raw = t['x'], t['c1'], t['raw']
            nvox = raw.buf[0, ..., 0].numel()
            dw1, db1, dg1, db1n, dw2, db2, dg2, db2n = slots[-8:]
            gy = _dense(torch.zeros(tuple(raw.buf.shape[:4]) + (c1.cout,), dtype=td, device=dev))   # pad channels stay 0
            (g1w, g1b), (g2w, g2b) = t['g1'], t['g2']
            for p in range(3):
                lib.call('seg3d_outblock_tail_bwd', dt, p, raw.p, raw.ld, nc, lib.ptr(t['s1']), lib.ptr(g1w), lib.ptr(g1b),
                         lib.ptr(t['w2']), lib.ptr(t['b2']), lib.ptr(t['s2']), lib.ptr(g2w), lib.ptr(g2b), GN_EPS, lib.ptr(gout),
                         lib.ptr(sums[-2]), lib.ptr(sums[-1]), lib.ptr(dg2), lib.ptr(db2n), lib.ptr(dw2), lib.ptr(db2),
                         lib.ptr(dg1), lib.ptr(db1n), lib.ptr(db1), gy.p, gy.ld, B, nvox, st())
            xd = x.buf.shape[1:4]
            lib.call('seg3d_conv3d_wgrad', lib.CONV_K3, dt, x.p, x.ld, c1.cin, gy.p, gy.ld, c1.cout, lib.ptr(dw1), B,
                     xd[0], xd[1], xd[2], st())
            dgrad = dgrad_of(t['conv1'], lib.CONV_K3, c1, x, xd, pad_cout=c1.cout if c1.cout != c1.real_cout else 0)
            if dgrad is not None:
                dcv, gd, od = dgrad
                lib.call('seg3d_conv3d_fwd', dcv.mode, dt, dcv.impl, gy.p, gy.ld, dcv.cin, lib.ptr(dcv.w), None,
                         gd.p, gd.ld, dcv.cout, B, od[0], od[1], od[2], None, st())
                add_contrib(x, gd)
            conv_grads(t['conv1'], lib.CONV_K3, c1, dw1, db1)
            grads[id(t['conv2'].weight)] = dw2.view(nc, nc, 1, 1, 1)
            grads[id(t['conv2'].bias)] = db2
            for holder, dgm, dbt in ((t['gn1'], dg1, db1n), (t['gn2'], dg2, db2n)):
                grads[id(holder.weight)], grads[id(holder.bias)] = dgm, dbt
        else:
            o = self.out
            g = torch.empty(tuple(o.buf.shape[:4]) + (o.C,), dtype=td, device=dev)
            lib.call('seg3d_grad_from_ncdhw', dt, lib.ptr(gout), o.C, B, g[0, ..., 0].numel(), lib.ptr(g), o.C, 0, st())
            contrib.setdefault((id(o.buf), o.off), []).append(_dense(g))

        # ---- conv -> GroupNorm units in reverse ------------------------------------------------------------------------
        for ui in range(len(self.units) - 1, -1, -1):
            u = self.units[ui]
            c, gn = u['c'], u['gn']
            gsrc = contrib.get((id(u['out'].buf), u['out'].off), [])
            assert 1 <= len(gsrc) <= 3, (ui, len(gsrc))
            gy = _dense(torch.empty(tuple(u['raw'].buf.shape[:4]) + (c.cout,), dtype=td, device=dev))
            dres = None if u['res'] is None else _dense(torch.empty_like(u['res'].buf))
            dw, db, dgm, dbt = slots[4 * ui:4 * ui + 4]
            dgrad = dgrad_of(u['conv'], u['mode'], c, u['x'], u['od'])
            gamma = gn.weight.detach().float().contiguous()
            beta = gn.bias.detach().float().contiguous()
            unit_step(dt, B, gsrc, u['out'], u['raw'], c.cout, lib.ptr(u['stats']), lib.ptr(gamma), lib.ptr(beta),
                      lib.ptr(sums[ui]), lib.ptr(dgm), lib.ptr(dbt), gy, dres, lib.ptr(db), u['od'].numel(), u['mode'], u['x'],
                      c.cin, lib.ptr(dw), u['xd'], dgrad, relu=u['relu'])
            if dres is not None:
                add_contrib(u['res'], dres)
            if dgrad is not None:
                add_contrib(u['x'], dgrad[1])
            conv_grads(u['conv'], u['mode'], c, dw, db)
            grads[id(gn.weight)], grads[id(gn.bias)] = dgm, dbt

        # ---- input gradients: the sum of each input's contributions, NCDHW fp32 -----------------------------------------
        din = {}
        for i, v in self.inputs.items():
            if not need_input[i]:
                continue
            gs = contrib.get((id(v.buf), v.off), [])
            assert 1 <= len(gs) <= 3, ('input', i, len(gs))
            B_, D, H, W, _ = v.buf.shape
            out = torch.empty((B_, v.C, D, H, W), dtype=torch.float32, device=dev)
            args = []
            for k in range(3):
                gk = gs[k] if k < len(gs) else None
                args += [lib.ptr(gk.buf), gk.ld, gk.off] if gk is not None else [None, 0, 0]
            lib.call('seg3d_grad_to_ncdhw', dt, len(gs), *args, v.C, B_, D * H * W, lib.ptr(out), st())
            din[i] = out
        return din, grads
