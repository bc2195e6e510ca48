"""Training forward/backward of the V-shaped networks on the C-ABI kernels (reference core/seg_train.py:122-124:
`outputs = net(crops); loss.backward()`).

Forward = the same kernel plan as inference, built in `train` mode so every pre-GroupNorm tensor and every
activation is kept.  Backward walks the recorded conv->GN->ReLU units in reverse, issuing only what autograd asks for
(_Backward.schedule: frozen weights get no weight gradient, a unit with nothing trainable at or upstream of it is skipped,
the network input gets a gradient when it requires one):

    gn_bwd pass 0/1  (dz = g*[out>0], GroupNorm backward, dgamma/dbeta/dbias, residual gradient)
    conv wgrad       (seg3d_conv3d_wgrad, fp32 accumulation)
    conv dgrad       (seg3d_conv3d_fwd on transformed weights: flipped k3, k2s2 <-> transposed conv)

An activation can have up to three consumers (next conv, residual add, skip connection); each consumer writes
its contribution into its own buffer and the producer's gn_bwd sums them on the fly, so nothing is accumulated
read-modify-write.  All arithmetic is in libseg3d_b200.so; torch only owns the buffers and the autograd node.
"""
import os

import torch

from . import dist as D
from . import lib
from .plan import GN_EPS, _Conv, _View


def _k3_dgrad_weight(w):        # [Co,Ci,3,3,3] -> conv weight of the data-gradient convolution [Ci,Co,3,3,3]
    return w.flip(2, 3, 4).permute(1, 0, 2, 3, 4).contiguous()


def _same_weight(w):            # k2s2 dgrad = transposed conv (and vice versa) on the very same tensor
    return w


_k3_dgrad_weight.seg3d_kind = 'k3_dgrad'       # index-map forms of these transforms: packing.py::add_conv_pack
_same_weight.seg3d_kind = 'identity'


def unit_step(dt, B, gsrc, out, raw, C, stats, gamma, beta, sums, dgamma, dbeta, gy, dres, dbias, nvox, mode, x, cin, dw, xd,
              dgrad=None, relu=True, xpad=None):
    """Backward of one conv -> GroupNorm [-> ReLU] [+ residual] unit, shared by the whole-network walk (_Backward.run) and
    the standalone modules (blocks.py):
        gn_bwd pass 0/1   dz = sum of the output's gradient contributions `gsrc` (1..3 _Views), masked by the ReLU when
                          `relu`; dy -> gy, dz -> dres (a unit with a residual), dgamma/dbeta/dbias
        conv wgrad        dw (kernel layout, fp32, accumulated) from the unit's input x (dims xd) and gy
        conv dgrad        dgrad = (dgrad convolution, gradient view, gy's dims), or None when no input gradient is needed
    dw=None skips the weight gradient (a frozen convolution).
    `xpad` (whole network only): the input block's row-padded input, whose weight gradient has a kernel of its own."""
    st = lib.stream_ptr
    gv = list(gsrc) + [None] * (3 - len(gsrc))
    g = (gv[0].p, gv[0].ld, gv[1].p if gv[1] else None, gv[1].ld if gv[1] else 0, gv[2].p if gv[2] else None, gv[2].ld if gv[2] else 0)
    if relu:
        # without a residual the ReLU mask is recomputed from the raw tensor the kernel reads anyway (out = NULL)
        remask = dres is None and os.environ.get('SEG3D_GN_BWD_REMASK', '1') != '0'
        for p in range(2):
            lib.call('seg3d_gn_bwd', dt, p, *g, None if remask else out.p, out.ld, raw.p, raw.ld, C, stats, gamma, beta, GN_EPS,
                     sums, dgamma, dbeta, gy.p, gy.ld, dres.p if dres else None, dres.ld if dres else 0, dbias, B, nvox, st())
    else:
        for p in range(2):
            lib.call('seg3d_gn_bwd_noact', dt, p, *g, raw.p, raw.ld, C, stats, gamma, GN_EPS,
                     sums, dgamma, dbeta, gy.p, gy.ld, dres.p if dres else None, dres.ld if dres else 0, dbias, B, nvox, st())
    if dw is None:
        pass
    elif xpad is not None:
        lib.call('seg3d_conv3d_cin1_wgrad', dt, xpad.p, xd[2] + lib.CIN1_PAD, gy.p, gy.ld, dw, B, xd[0], xd[1], xd[2], st())
    else:
        lib.call('seg3d_conv3d_wgrad', mode, dt, x.p, x.ld, cin, gy.p, gy.ld, C, dw, B, xd[0], xd[1], xd[2], st())
    if dgrad is not None:
        dcv, gd, od = dgrad
        lib.call('seg3d_conv3d_fwd', dcv.mode, dt, dcv.impl, gy.p, gy.ld, dcv.cin, lib.ptr(dcv.w), None,
                 gd.p, gd.ld, dcv.cout, B, od[0], od[1], od[2], None, st())


class _Backward(object):
    """Per (plan, shape) backward state: gradient buffers, dgrad convolutions, parameter-gradient slots."""

    def __init__(self, plan, ws):
        self.plan, self.ws = plan, ws
        dev, td = plan.device, plan.tdtype
        B, vox = ws['B'], ws['vox']
        self.units = ws['units']
        self.gy, self.gd, self.dres = {}, {}, {}
        self.dconv = {}
        self.produced = {}                    # (id(buf), off) -> producing unit's out view
        for u in self.units:
            self.produced[(id(u['out'].buf), u['out'].off)] = u['out']
        # parameter gradients in kernel layouts: fp32 views into ONE flat buffer, zeroed with a single memset per step
        sizes = []
        for u in self.units:
            c = plan.convs[u['conv']]
            C = c.cout
            self.gy[u['conv']] = _View(torch.empty((B, vox[u['lout']], C), dtype=td, device=dev), 0, C, C)
            if u['res'] is not None:
                r = u['res']
                self.dres[u['conv']] = _View(torch.empty((B, vox[u['lout']], r.C), dtype=td, device=dev), 0, r.C, r.C)
            if self._has_producer(u['x']):
                self.gd[u['conv']] = _View(torch.empty((B, vox[u['lin']], u['x'].C), dtype=td, device=dev), 0, u['x'].C, u['x'].C)
            taps = {lib.CONV_K3: 27, lib.CONV_K2S2: 8, lib.CONV_T2S2: 8}[c.mode]
            sizes += [(u['conv'] + '.weight', taps * c.cin * c.cout), (u['conv'] + '.bias', c.cout),
                      (u['gn'] + '.weight', c.cout), (u['gn'] + '.bias', c.cout)]
        nc = plan.out_channels
        c1 = plan.convs['out_block.conv1']
        # when conv1 runs zero-padded to 16 output channels on the tensor cores, its weight gradient does too
        self.conv1_co = c1.cout
        sizes += [('out_block.conv1.weight', 27 * c1.cin * self.conv1_co),
                  ('out_block.conv1.bias', nc), ('out_block.gn1.weight', nc), ('out_block.gn1.bias', nc),
                  ('out_block.conv2.weight', nc * nc), ('out_block.conv2.bias', nc),
                  ('out_block.gn2.weight', nc), ('out_block.gn2.bias', nc)]
        total = sum((n + 3) // 4 * 4 for _, n in sizes)          # 16-byte aligned slots
        self.pgrad_flat = torch.zeros((total,), dtype=torch.float32, device=dev)
        self.pgrad, self.pg_off, off = {}, {}, 0
        for k, n in sizes:
            self.pgrad[k] = self.pgrad_flat[off:off + n]
            self.pg_off[k] = off
            off += (n + 3) // 4 * 4
        self.pg_total = off
        self.grads_reduced = False
        ncp = ws['tail']['ncp']
        self.gy_tail = _View(torch.zeros((B, vox[0], ncp), dtype=td, device=dev), 0, ncp, ncp)   # pad channels stay 0
        tx = ws['tail']['x']
        self.gd_tail = _View(torch.empty((B, vox[0], tx.C), dtype=td, device=dev), 0, tx.C, tx.C)
        self.sums = torch.zeros((len(self.units) + 2, B, 2), dtype=torch.float64, device=dev)
        self.schedules = {}
        self.dconv_in, self.gd_in = None, None      # multi-channel input gradient, built when first asked for (_input_dgrad)
        self._make_dgrad_convs()
        self._make_tables()

    def _has_producer(self, x):
        return any(id(x.buf) == k[0] and x.off <= k[1] < x.off + x.C for k in self.produced)

    def _inside(self, xv):
        """keys of the producers inside consumer input window xv (the channel-span rule of add_contrib)"""
        return [(bid, off) for (bid, off), pv in self.produced.items()
                if bid == id(xv.buf) and xv.off <= off and off + pv.C <= xv.off + xv.C]

    def schedule(self, need_input, need):
        """What the walk issues for one gradient mask (need_input: the network input needs a gradient; need: the names of
        the parameters that do), cached per mask.  A unit is needed when one of its parameters is trainable or a producer
        inside its input (or residual) window is needed - for the input block, when the input needs a gradient.  A unit that
        is not needed issues nothing; a needed one runs both GroupNorm backward passes, its weight gradient only when its
        conv weight or bias is trainable, and its data gradient only when its input needs one.  The out-block tail follows
        the same rule.  Returns {'units': [(run, wgrad, dgrad)], 'tail': (run, wgrad, dgrad), 'slots': (lo, hi)}, where
        [lo, hi) is the range of the flat parameter-gradient buffer that holds the trainable parameters."""
        key = (bool(need_input), frozenset(need))
        sched = self.schedules.get(key)
        if sched is not None:
            return sched
        needed, units = {}, []
        for u in self.units:
            conv_t = u['conv'] + '.weight' in need or u['conv'] + '.bias' in need
            gn_t = u['gn'] + '.weight' in need or u['gn'] + '.bias' in need
            if u['conv'] == 'in_block.conv':
                dgrad = bool(need_input)
            else:
                dgrad = any(needed[k] for k in self._inside(u['x']))
            res = u['res'] is not None and any(needed[k] for k in self._inside(u['res']))
            run = conv_t or gn_t or dgrad or res
            needed[(id(u['out'].buf), u['out'].off)] = run
            units.append((run, run and conv_t, dgrad))
        tail_t = any(k.startswith('out_block.') for k in need)
        tail_dgrad = any(needed[k] for k in self._inside(self.ws['tail']['x']))
        tail_w = 'out_block.conv1.weight' in need or 'out_block.conv1.bias' in need
        tail_run = tail_t or tail_dgrad
        ends = [(self.pg_off[k], self.pg_off[k] + self.pgrad[k].numel()) for k in need if k in self.pg_off]
        slots = (min(a for a, _ in ends), max(b for _, b in ends)) if ends else (0, 0)
        sched = self.schedules[key] = {'units': units, 'tail': (tail_run, tail_run and tail_w, tail_dgrad), 'slots': slots}
        return sched

    def _make_dgrad_convs(self):
        plan = self.plan
        sd = self._weights()
        for name, c in list(plan.convs.items()):
            if name == 'in_block.conv':     # the network input's gradient: _input_grad
                continue
            if c.mode == lib.CONV_K3:
                pad = c.cout if c.cout != c.real_cout else 0
                self.dconv[name] = _Conv(sd, name, lib.CONV_K3, plan.dt, plan.device, plan.tc_modes,
                                         transform=_k3_dgrad_weight, pad_dim0=pad)
            elif c.mode == lib.CONV_K2S2:    # dgrad of the stride-2 conv = transposed conv with the same tensor
                self.dconv[name] = _Conv(sd, name, lib.CONV_T2S2, plan.dt, plan.device, plan.tc_modes, transform=_same_weight)
            else:                            # dgrad of the transposed conv = stride-2 conv with the same tensor
                self.dconv[name] = _Conv(sd, name, lib.CONV_K2S2, plan.dt, plan.device, plan.tc_modes, transform=_same_weight)

    def _weights(self):
        return self.plan._last_sd

    def _make_tables(self):
        """one-launch re-pack of the data-gradient weights and one-launch un-pack of the weight gradients (packing.py), when the
        plan is bound to the live parameter tensors"""
        from . import packing
        plan = self.plan
        self.pack_table, self.unpack_table, self.gflat = None, None, None
        if not plan._bound_valid():
            return
        named = plan.bound
        t = packing.PackTable(plan.device)
        for name, c in self.dconv.items():
            packing.add_conv_pack(t, c, named[name + '.weight'].data, None)
        self.pack_table = t
        # kernel-layout gradient slots -> one flat buffer in parameter layout and order
        offsets, total = packing.flat_layout(list(named.items()))
        self.gflat = torch.zeros((total,), dtype=torch.float32, device=plan.device)
        self.g_offsets, self.g_shapes = offsets, {k: tuple(v.shape) for k, v in named.items()}
        u = packing.PackTable(plan.device)
        for name, c in plan.convs.items():
            slot = self.pgrad[name + '.weight']
            co_slot = self.conv1_co if name == 'out_block.conv1' else c.cout
            P0, P1, k = self.g_shapes[name + '.weight'][:3]
            base = offsets[name + '.weight']
            if c.mode == lib.CONV_T2S2:          # slot [Cin][tap][Cout] -> parameter [Cin][Cout][a][b][c]
                sstride = [8 * co_slot, 1, 4 * co_slot, 2 * co_slot, co_slot]
            else:                                # slot [tap][Cin][Cout] -> parameter [Cout][Cin][a][b][c]
                sstride = [1, co_slot, k * k * P1 * co_slot, k * P1 * co_slot, P1 * co_slot]
            u.add(self.pgrad_flat, self.gflat, [P0, P1, k, k, k], sstride, [P1 * k ** 3, k ** 3, k * k, k, 1],
                  src_base=self.pg_off[name + '.weight'], dst_base=base)
            nb = self.g_shapes[name + '.bias'][0]
            u.add(self.pgrad_flat, self.gflat, [1, 1, 1, 1, nb], [0, 0, 0, 0, 1], [0, 0, 0, 0, 1],
                  src_base=self.pg_off[name + '.bias'], dst_base=offsets[name + '.bias'])
        for key in ('out_block.conv2.weight', 'out_block.conv2.bias'):
            n = 1
            for d in self.g_shapes[key]:
                n *= d
            u.add(self.pgrad_flat, self.gflat, [1, 1, 1, 1, n], [0, 0, 0, 0, 1], [0, 0, 0, 0, 1],
                  src_base=self.pg_off[key], dst_base=offsets[key])
        for name in plan.gns:
            for leaf in ('.weight', '.bias'):
                n = self.g_shapes[name + leaf][0]
                u.add(self.pgrad_flat, self.gflat, [1, 1, 1, 1, n], [0, 0, 0, 0, 1], [0, 0, 0, 0, 1],
                      src_base=self.pg_off[name + leaf], dst_base=offsets[name + leaf])
        self.unpack_table = u

    def refresh(self):
        if self.dconv_in is not None:
            self.dconv_in.load(self._weights())
        if self.pack_table is not None and self.plan._bound_valid():
            self.pack_table.run()
            return
        sd = self._weights()
        for c in self.dconv.values():
            c.load(sd)

    def _input_dgrad(self):
        """(dgrad convolution, gradient view, gy dims) of a multi-channel network input's gradient, built on first use so that
        a step that does not ask for it re-packs and allocates nothing for it"""
        plan, ws = self.plan, self.ws
        if self.dconv_in is None:
            self.dconv_in = _Conv(self._weights(), 'in_block.conv', lib.CONV_K3, plan.dt, plan.device, plan.tc_modes,
                                  transform=_k3_dgrad_weight)
            C = plan.in_channels
            self.gd_in = _View(torch.empty((ws['B'], ws['vox'][0], C), dtype=plan.tdtype, device=plan.device), 0, C, C)
        return self.dconv_in, self.gd_in, ws['dims'][0]

    # --------------------------------------------------------------------------------------------
    def run(self, dprobs, need_input=False, need=None):
        """-> (parameter gradients by name, input gradient or None).  need: the parameter names that need a gradient
        (None: every parameter); the gradients of the others are not computed and must not be used."""
        plan, ws = self.plan, self.ws
        if need is None:
            need = self.pgrad.keys()
        sched = self.schedule(need_input, need)
        slot_lo, slot_hi = sched['slots']
        B, vox, dims, dt = ws['B'], ws['vox'], ws['dims'], plan.dt
        st = lib.stream_ptr
        self.pgrad_flat.zero_()
        self.sums.zero_()
        contrib = {}
        # data parallel: the slots are laid out in forward order and the walk below finishes them back to front, so the
        # finished tail of the flat buffer is all-reduced (NCCL, its own stream) while the rest of the backward pass runs.
        # Only the slots of trainable parameters, [slot_lo, slot_hi), are reduced.
        _, world = D.world()
        overlap = world > 1 and os.environ.get('SEG3D_OVERLAP_ALLREDUCE', '1') != '0'
        works, sent_lo = [], slot_hi
        bucket = int(os.environ.get('SEG3D_ALLREDUCE_BUCKET_MB', '12')) << 18          # floats

        def reduce_tail(lo, force=False):
            nonlocal sent_lo
            lo = max(lo, slot_lo)
            if overlap and sent_lo > lo and (force or sent_lo - lo >= bucket):
                works.append(torch.distributed.all_reduce(self.pgrad_flat[lo:sent_lo], op=torch.distributed.ReduceOp.SUM,
                                                          async_op=True))
                sent_lo = lo

        def add_contrib(xv, gv):
            """register gradient view gv (same channel span as consumer input xv) with every producer inside xv"""
            for (bid, off), pv in self.produced.items():
                if bid == id(xv.buf) and xv.off <= off and off + pv.C <= xv.off + xv.C:
                    sub = _View(gv.buf, gv.off + (off - xv.off), gv.ld, pv.C)
                    contrib.setdefault((bid, off), []).append(sub)

        # ---- output block tail -----------------------------------------------------------------
        nc = plan.out_channels
        tail = ws['tail']
        g1, g2 = plan.gns['out_block.gn1'], plan.gns['out_block.gn2']
        s1 = lib.ptr(ws['stats'][plan.gn_index['out_block.gn1']])
        s2 = lib.ptr(ws['stats2'])
        nu = len(self.units)
        sums2, sums1 = lib.ptr(self.sums[nu]), lib.ptr(self.sums[nu + 1])
        pg = self.pgrad
        dp = dprobs.contiguous().float()
        tail_run, tail_w, tail_dgrad = sched['tail']
        for p in range(3 if tail_run else 0):
            lib.call('seg3d_outblock_tail_bwd', dt, p, tail['raw'].p, tail['raw'].ld, nc, s1, lib.ptr(g1.gamma), lib.ptr(g1.beta),
                     lib.ptr(plan.w2), lib.ptr(plan.b2), s2, lib.ptr(g2.gamma), lib.ptr(g2.beta), GN_EPS, lib.ptr(dp),
                     sums2, sums1, lib.ptr(pg['out_block.gn2.weight']), lib.ptr(pg['out_block.gn2.bias']),
                     lib.ptr(pg['out_block.conv2.weight']), lib.ptr(pg['out_block.conv2.bias']),
                     lib.ptr(pg['out_block.gn1.weight']), lib.ptr(pg['out_block.gn1.bias']), lib.ptr(pg['out_block.conv1.bias']),
                     self.gy_tail.p, self.gy_tail.ld, B, vox[0], st())
        x = tail['x']
        d0 = dims[0]
        if tail_w:
            lib.call('seg3d_conv3d_wgrad', lib.CONV_K3, dt, x.p, x.ld, x.C, self.gy_tail.p, self.gy_tail.ld, self.conv1_co,
                     lib.ptr(pg['out_block.conv1.weight']), B, d0[0], d0[1], d0[2], st())
        if tail_dgrad:
            dc = self.dconv['out_block.conv1']
            lib.call('seg3d_conv3d_fwd', lib.CONV_K3, dt, dc.impl, self.gy_tail.p, self.gy_tail.ld, dc.cin, lib.ptr(dc.w), None,
                     self.gd_tail.p, self.gd_tail.ld, dc.cout, B, d0[0], d0[1], d0[2], None, st())
            add_contrib(x, self.gd_tail)
        reduce_tail(self.pg_off['out_block.conv1.weight'])

        # ---- conv -> GN -> ReLU units in reverse ---------------------------------------------------
        dx = None
        for ui in range(nu - 1, -1, -1):
            u = self.units[ui]
            run, wgrad, need_dgrad = sched['units'][ui]
            if not run:
                continue
            c = plan.convs[u['conv']]
            gsrc = contrib.get((id(u['out'].buf), u['out'].off), [])
            assert 1 <= len(gsrc) <= 3, (u['conv'], len(gsrc))
            gnp = plan.gns[u['gn']]
            sf = lib.ptr(ws['stats'][plan.gn_index[u['gn']]])
            gy = self.gy[u['conv']]
            dres = self.dres.get(u['conv'])
            dgrad = None
            if need_dgrad and u['conv'] in self.gd:    # the dgrad convolution's input is dy, living at the unit's output level
                dgrad = (self.dconv[u['conv']], self.gd[u['conv']], dims[u['lout']])
            elif need_dgrad and u['conv'] == 'in_block.conv' and plan.in_channels > 1:
                dgrad = self._input_dgrad()
            # input block on the row-padded input (Toeplitz operands)
            xpad = u['xpad'] if u.get('xpad') is not None and gy.ld == 16 else None
            unit_step(dt, B, gsrc, u['out'], u['raw'], c.cout, sf, lib.ptr(gnp.gamma), lib.ptr(gnp.beta), lib.ptr(self.sums[ui]),
                      lib.ptr(pg[u['gn'] + '.weight']), lib.ptr(pg[u['gn'] + '.bias']), gy, dres, lib.ptr(pg[u['conv'] + '.bias']),
                      vox[u['lout']], c.mode, u['x'], c.cin, lib.ptr(pg[u['conv'] + '.weight']) if wgrad else None,
                      dims[u['lin']], dgrad, xpad=xpad)
            if dres is not None:
                add_contrib(u['res'], dres)
            if u['conv'] == 'in_block.conv' and need_dgrad:
                dx = self._input_grad(gy, dgrad)
            elif dgrad is not None:
                add_contrib(u['x'], dgrad[1])
            reduce_tail(self.pg_off[u['conv'] + '.weight'])
        reduce_tail(slot_lo, force=True)
        for w in works:
            w.wait()
        self.grads_reduced = bool(works)
        if works:
            self.pgrad_flat.mul_(1.0 / world)
        return self._param_grads(), dx

    def _input_grad(self, gy, dgrad):
        """NCDHW fp32 gradient of the network input from the input block's conv-output gradient gy: one
        seg3d_conv3d_cin1_dgrad for a single-channel input, else the generic data-gradient convolution (already issued by
        unit_step into dgrad's view) turned into NCDHW by seg3d_grad_to_ncdhw.  It is not part of the flat parameter buffer."""
        plan, ws = self.plan, self.ws
        B, (D, H, W) = ws['B'], ws['dims'][0]
        dx = torch.empty((B, plan.in_channels, D, H, W), dtype=torch.float32, device=plan.device)
        if plan.in_channels == 1:
            lib.call('seg3d_conv3d_cin1_dgrad', plan.dt, gy.p, gy.ld, lib.ptr(plan.convs['in_block.conv'].w), lib.ptr(dx),
                     B, D, H, W, lib.stream_ptr())
        else:
            gd = dgrad[1]
            lib.call('seg3d_grad_to_ncdhw', plan.dt, 1, lib.ptr(gd.buf), gd.ld, gd.off, None, 0, 0, None, 0, 0, plan.in_channels,
                     B, D * H * W, lib.ptr(dx), lib.stream_ptr())
        return dx

    def _param_grads(self):
        """kernel-layout fp32 gradients -> the reference's parameter layouts: one seg3d_gather_pack launch into a flat buffer
        in parameter order, handed to autograd as views of ONE fresh copy (the slots are rewritten next step; the optimiser of
        _b200/optim.py recognises the flat buffer and updates every parameter with one launch)."""
        if self.unpack_table is not None and self.plan._bound_valid():
            self.unpack_table.run()
            flat = self.gflat.clone()
            out = {}
            for name, shape in self.g_shapes.items():
                n = 1
                for d in shape:
                    n *= d
                out[name] = flat[self.g_offsets[name]:self.g_offsets[name] + n].view(shape)
            return out
        plan, out = self.plan, {}
        for name, c in plan.convs.items():
            g = self.pgrad[name + '.weight']
            if c.mode == lib.CONV_T2S2:
                out[name + '.weight'] = g.view(c.cin, 2, 2, 2, c.cout).permute(0, 4, 1, 2, 3)
            else:
                k = 3 if c.mode == lib.CONV_K3 else 2
                out[name + '.weight'] = g.view(k, k, k, c.cin, c.cout)[..., :c.real_cout].permute(4, 3, 0, 1, 2)
            out[name + '.bias'] = self.pgrad[name + '.bias'][:c.real_cout]
        nc = plan.out_channels
        out['out_block.conv2.weight'] = self.pgrad['out_block.conv2.weight'].view(nc, nc, 1, 1, 1)
        out['out_block.conv2.bias'] = self.pgrad['out_block.conv2.bias']
        for name in plan.gns:
            out[name + '.weight'] = self.pgrad[name + '.weight'][:nc] if name.startswith('out_block') else self.pgrad[name + '.weight']
            out[name + '.bias'] = self.pgrad[name + '.bias'][:nc] if name.startswith('out_block') else self.pgrad[name + '.bias']
        return out


class _NetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, x, names, *params):
        plan = net._current_plan(train=True)
        B, Cin, D, H, W = x.shape
        ws, ops = plan.plan(B, D, H, W, train=True)
        plan.load_input(ws, x.detach().float())
        probs = plan.run(ws, ops).clone()
        # the saved activations live in the plan's workspace, shared by every forward of this shape: stamp the forward so
        # that a backward after a LATER forward of the same shape (gradient accumulation over two crops, two forwards
        # before one backward) fails loudly instead of differentiating the wrong activations
        ws['generation'] = ws.get('generation', 0) + 1
        ctx.plan, ctx.ws, ctx.names, ctx.generation = plan, ws, names, ws['generation']
        return probs

    @staticmethod
    def backward(ctx, dprobs):
        plan, ws = ctx.plan, ctx.ws
        if ws.get('generation') != ctx.generation:
            raise RuntimeError('seg3d_b200: the activations of this forward were overwritten by a later forward of the same '
                               'shape; call backward() before the next forward (one forward per backward)')
        bw = ws.get('bwd')
        if bw is None:
            bw = ws['bwd'] = _Backward(plan, ws)
        else:
            bw.refresh()
        need = {n for n, f in zip(ctx.names, ctx.needs_input_grad[3:]) if f}
        grads, dx = bw.run(dprobs, ctx.needs_input_grad[1], need)
        plan.grads_reduced_in_backward = bw.grads_reduced       # train_step then skips its own all-reduce
        # the slots are reused next step: hand autograd its own copy (one copy, in the reference's parameter layout);
        # frozen parameters get None
        if bw.unpack_table is not None:
            return (None, dx, None) + tuple(grads[n] if n in need else None for n in ctx.names)   # views of a private flat copy
        return (None, dx, None) + tuple((g.clone() if g.is_contiguous() else g.contiguous()) if n in need else None
                                        for n, g in ((n, grads[n]) for n in ctx.names))


def train_forward(net, x):
    names = [n for n, _ in net.named_parameters()]
    params = [p for _, p in net.named_parameters()]
    return _NetFunction.apply(net, x, names, *params)
