"""Forward plan of VNet / VBNet on the C-ABI kernels.

Host-side plumbing only: packs the reference-layout fp32 weights (OIDHW / IODHW) into the kernel
layouts, owns the NDHWC workspaces (torch tensors = device memory), and issues the kernel
sequence that restates SegmentationNet.forward (reference network/vnet.py:36-48, vbnet.py:38-50).
All arithmetic happens in libseg3d_b200.so.

Data layout in HBM (per forward of B patches of D x H x W):
  * activations NDHWC, storage dtype = the plan's mode (fp32 strict / fp16 / bf16);
  * skip tensors live inside their concat buffers from the moment they are produced
    (channel offset + pitch), so torch.cat (vnet_upblock.py:21) never runs;
  * one `raw` scratch holds each convolution's pre-GroupNorm result until the next
    seg3d_gn_apply consumes it;
  * one double[n_gn][B][2] tensor carries the GroupNorm partial sums.
"""
import os

import torch

from . import lib

# 'fp32x': strict parity on the tensor cores - f16 storage of split operands (x = hi + lo), three MMAs per product
MODES = {'fp32': lib.F32, 'fp16': lib.F16, 'bf16': lib.BF16, 'fp32x': lib.F16}
GN_EPS = 1e-5


def _require_cuda(device, message):
    """The product runs on CUDA devices only.  A function of its own so that the host-wiring tests of the CPU gate
    (tests/test_plan_wiring.py: C-ABI calls emulated, CPU tensors) can stub it; nothing in the package does."""
    if device.type != 'cuda':
        raise RuntimeError(message)


def detect_arch(sd):
    return 'vbnet' if any('.conv1.conv.weight' in k for k in sd) else 'vnet'


def strip_prefix(sd):
    if any(k.startswith('module.') for k in sd):
        return {k[7:]: v for k, v in sd.items()}
    return dict(sd)


class _Conv(object):
    """One packed convolution.  `load` (re)packs in place so kernel-argument pointers stay valid."""

    def __init__(self, sd, name, mode, dt, device, allow_tc, pad_cout=0, transform=None, pad_dim0=0, fold=False, split=False):
        self.transform, self.pad_dim0 = transform, pad_dim0
        self.fold, self.w_fold = fold, None
        self.split = split          # strict mode on the tensor cores: weights packed [.. Cout][whi(Cin) | wlo(Cin)] f16
        w = self._effective_weight(sd[name + '.weight'])
        self.name, self.mode, self.dt, self.device = name, mode, dt, device
        if mode == lib.CONV_T2S2:
            self.cin, self.cout = w.shape[0], w.shape[1]
        else:
            self.cout, self.cin = w.shape[0], w.shape[1]
        # pad_cout: zero-pad the output channels (weights and bias) so a narrow conv (out_block.conv1,
        # Cout = classes) can run on the tensor cores, whose minimum N is 16 at M=128.  The padded
        # channels are exactly 0, so they add nothing to the GroupNorm sums.
        self.real_cout = self.cout
        if pad_cout and allow_tc and dt != lib.F32 and mode in allow_tc and self.cout < pad_cout:
            self.cout = pad_cout
        tc_ok = (allow_tc and dt != lib.F32 and self.cin % 16 == 0 and self.cout % 16 == 0 and self.cout <= 256
                 and mode in allow_tc)
        self.impl = lib.IMPL_TCGEN05 if tc_ok else lib.IMPL_SIMT
        # input block (Cin == 1): the tensor-core kernel builds its own im2col tile and takes the fp32 SIMT weight
        # layout, so packing follows `impl` (SIMT) while the call lets the library pick (csrc/conv_tc_cin1.cu)
        self.cin1_tc = bool(not tc_ok and allow_tc and dt != lib.F32 and not split and mode == lib.CONV_K3 and mode in allow_tc
                            and self.cin == 1 and self.cout == 16 and transform is None)
        self.call_impl = lib.IMPL_AUTO if self.cin1_tc else self.impl
        self.w, self.bias = None, None
        self.load(sd)

    def _effective_weight(self, w):
        """dgrad convolutions reuse the forward kernels on a transformed view of the same parameter."""
        w = w.detach()
        if self.pad_dim0 and w.shape[0] < self.pad_dim0:
            wp = torch.zeros((self.pad_dim0,) + tuple(w.shape[1:]), dtype=w.dtype, device=w.device)
            wp[:w.shape[0]] = w
            w = wp
        return self.transform(w) if self.transform is not None else w

    def load(self, sd):
        w = self._effective_weight(sd[self.name + '.weight']).to(device=self.device, dtype=torch.float32)
        b = sd.get(self.name + '.bias') if self.transform is None and not self.pad_dim0 else None
        if self.cout != self.real_cout:
            wp = torch.zeros((self.cout,) + tuple(w.shape[1:]), dtype=torch.float32, device=self.device)
            wp[:self.real_cout] = w
            w = wp
            if b is not None:
                bp = torch.zeros((self.cout,), dtype=torch.float32, device=self.device)
                bp[:self.real_cout] = b.detach().to(self.device)
                b = bp
        if self.impl == lib.IMPL_SIMT:
            if self.mode == lib.CONV_T2S2:      # [Cin][8*Cout], column = tap*Cout + co
                p = w.permute(0, 2, 3, 4, 1).reshape(self.cin, 8 * self.cout)
            else:                               # [taps][Cin][Cout]
                p = w.permute(2, 3, 4, 1, 0).reshape(-1, self.cin, self.cout)
            p = p.contiguous()
        elif self.split:
            if self.mode == lib.CONV_T2S2:      # [8*Cout][Cin]
                q = w.permute(2, 3, 4, 1, 0).reshape(8 * self.cout, self.cin)
            else:                               # [taps][Cout][Cin]
                q = w.permute(2, 3, 4, 0, 1).reshape(-1, self.cout, self.cin)
            hi = q.to(torch.float16)
            lo = (q - hi.float()).to(torch.float16)
            p = torch.cat([hi, lo], dim=-1).contiguous()
        else:
            if self.mode == lib.CONV_T2S2:      # [8*Cout][Cin]
                p = w.permute(2, 3, 4, 1, 0).reshape(8 * self.cout, self.cin)
            else:                               # [taps][Cout][Cin]
                p = w.permute(2, 3, 4, 0, 1).reshape(-1, self.cout, self.cin)
            p = p.contiguous().to(lib.TORCH_DTYPE[self.dt])
        if self.fold:
            # narrow-output k3 conv (seg3d_conv3d_k3_narrow_fwd): [kd][(kh,kw,co)][ci], rows zero-padded to NP
            C = self.real_cout
            NP = lib.load().seg3d_conv3d_k3_narrow_np(C)
            wf = torch.zeros((3, NP, self.cin), dtype=torch.float32, device=self.device)
            wf[:, :9 * C] = w[:C].permute(2, 3, 4, 0, 1).reshape(3, 9 * C, self.cin)
            if self.split:              # rows [whi(Cin) | wlo(Cin)] (seg3d_conv3d_k3_narrow_split_fwd)
                fhi = wf.to(torch.float16)
                wf = torch.cat([fhi, (wf - fhi.float()).to(torch.float16)], dim=-1).contiguous()
            else:
                wf = wf.to(lib.TORCH_DTYPE[self.dt]).contiguous()
            if self.w_fold is None:
                self.w_fold = wf
            else:
                self.w_fold.copy_(wf)
        if self.w is None:
            self.w = p
            self.bias = None if b is None else b.detach().to(device=self.device, dtype=torch.float32).contiguous()
        else:
            self.w.copy_(p)
            if b is not None:
                self.bias.copy_(b.detach())


class _GN(object):
    def __init__(self, sd, name, device):
        self.name = name
        self.gamma = sd[name + '.weight'].detach().to(device=device, dtype=torch.float32).contiguous().clone()
        self.beta = sd[name + '.bias'].detach().to(device=device, dtype=torch.float32).contiguous().clone()

    def load(self, sd):
        self.gamma.copy_(sd[self.name + '.weight'].detach())
        self.beta.copy_(sd[self.name + '.bias'].detach())


class _View(object):
    """Channel window [off, off+C) of an NDHWC buffer with pitch ld.  `sample` = elements per sample (0: unknown, whole-batch
    use only); `scratch`: a per-launch scratch (the raw pre-GroupNorm tensor) that every sub-batch of a schedule places at the
    start of the buffer, so consecutive sub-batches reuse the same, L2-resident addresses."""
    __slots__ = ('buf', 'off', 'ld', 'C', 'sample', 'scratch')

    def __init__(self, buf, off, ld, C, sample=0, scratch=False):
        self.buf, self.off, self.ld, self.C, self.sample, self.scratch = buf, off, ld, C, sample, scratch

    @property
    def p(self):
        return lib.ptr(self.buf, self.off)

    def at(self, b0):
        """pointer of sample b0"""
        if b0 == 0 or self.scratch:
            return lib.ptr(self.buf, self.off)
        assert self.sample > 0
        return lib.ptr(self.buf, self.off + b0 * self.sample)


class NetPlan(object):
    def __init__(self, state_dict, mode='fp16', device=None, arch=None, tc_modes=None):
        lib.load()
        if mode not in MODES:
            raise ValueError('mode must be one of %s' % sorted(MODES))
        self.mode, self.dt = mode, MODES[mode]
        self.split = mode == 'fp32x'
        self.in_dt = lib.F32 if self.split else self.dt      # storage type of the network input (patch gather output)
        self.tdtype = lib.TORCH_DTYPE[self.dt]
        self.device = torch.device(device if device is not None else 'cuda')
        _require_cuda(self.device, 'seg3d_b200 runs on CUDA devices only (no CPU fallback)')
        sd = strip_prefix(state_dict)
        self._last_sd = sd
        self.arch = arch or detect_arch(sd)
        if tc_modes is None:
            tc_modes = () if os.environ.get('SEG3D_FORCE_SIMT') == '1' else DEFAULT_TC_MODES
        self.tc_modes = tuple(tc_modes)
        self.in_channels = sd['in_block.conv.weight'].shape[1]
        self.out_channels = sd['out_block.conv2.weight'].shape[0]
        if self.out_channels > WIDE_MAX_CLASSES:
            raise RuntimeError('seg3d_b200: at most %d output classes are supported: the label mask is int8 '
                               '(seg3d_blend_finalize_argmax_z)' % WIDE_MAX_CLASSES)
        # more than 16 classes: the tensor-core tail (csrc/tail_wide.cu) on conv1's raw result, zero-padded to `wide_cp`
        # output channels and stored in fp32; up to 16 the SIMT tail stays the exact-fp32 path
        self.wide = self.out_channels > 16
        self.wide_cp = (self.out_channels + 15) // 16 * 16
        self.convs, self.gns = {}, {}
        for k in sd:
            if not k.endswith('.weight'):
                continue
            name = k[:-7]
            if sd[k].dim() == 5:
                if name.endswith('up_conv'):
                    m = lib.CONV_T2S2
                elif name.endswith('down_conv'):
                    m = lib.CONV_K2S2
                elif name == 'out_block.conv2':
                    continue
                else:
                    m = lib.CONV_K3
                narrow = (name == 'out_block.conv1' and self.dt != lib.F32 and lib.CONV_K3 in self.tc_modes
                          and sd[k].shape[0] <= 7 and sd[k].shape[1] in ((32,) if self.split else (16, 32, 64))
                          and os.environ.get('SEG3D_NARROW', '1') != '0')
                pad = (self.wide_cp if self.wide else 16) if name == 'out_block.conv1' else 0
                self.convs[name] = _Conv(sd, name, m, self.dt, self.device, self.tc_modes,
                                         pad_cout=pad, fold=narrow, split=self.split)
            else:
                self.gns[name] = _GN(sd, name, self.device)
        self.w2 = sd['out_block.conv2.weight'].detach().to(self.device, torch.float32).reshape(
            self.out_channels, self.out_channels).contiguous()
        self.b2 = sd['out_block.conv2.bias'].detach().to(self.device, torch.float32).contiguous()
        self.w2 = self.w2.clone()
        self.b2 = self.b2.clone()
        self.gn_names = sorted(self.gns)
        self.gn_index = {n: i for i, n in enumerate(self.gn_names)}
        self._plans = {}
        self.bound, self.pack_table = None, None
        self.launches_per_forward = 0
        self.use_graph = os.environ.get('SEG3D_GRAPH', '0') == '1'

    def bind_parameters(self, named_params):
        """Tie the plan to the live parameter tensors (fp32, contiguous, on the plan's device): `refresh` then re-packs every
        weight with ONE seg3d_gather_pack launch reading the parameters in place, instead of ~130 framework launches."""
        from . import packing
        named = {(k[7:] if k.startswith('module.') else k): v for k, v in named_params}
        ok = all(v.dtype == torch.float32 and v.is_contiguous() and v.device == self.device for v in named.values())
        if not ok or os.environ.get('SEG3D_PACK_KERNEL', '1') == '0':
            self.bound, self.pack_table = None, None
            return
        t = packing.PackTable(self.device)
        for name, c in self.convs.items():
            packing.add_conv_pack(t, c, named[name + '.weight'].data, named[name + '.bias'].data if (name + '.bias') in named else None)
        for name, g in self.gns.items():
            t.add_copy(named[name + '.weight'].data, g.gamma)
            t.add_copy(named[name + '.bias'].data, g.beta)
        t.add_copy(named['out_block.conv2.weight'].data, self.w2)
        t.add_copy(named['out_block.conv2.bias'].data, self.b2)
        self.bound = named
        self.bound_ptrs = {k: v.data_ptr() for k, v in named.items()}
        self.pack_table = t

    def _bound_valid(self):
        return getattr(self, 'bound', None) is not None and all(v.data_ptr() == self.bound_ptrs[k] for k, v in self.bound.items())

    def refresh(self, state_dict):
        """Re-pack changed weights in place (pointers captured by cached plans stay valid)."""
        sd = strip_prefix(state_dict)
        self._last_sd = sd
        if self._bound_valid():
            self.pack_table.run()
            return
        for c in self.convs.values():
            c.load(sd)
        for g in self.gns.values():
            g.load(sd)
        self.w2.copy_(sd['out_block.conv2.weight'].detach().reshape(self.out_channels, self.out_channels))
        self.b2.copy_(sd['out_block.conv2.bias'].detach())

    # ------------------------------------------------------------------------------------
    def _rblock_len(self, prefix):
        n = 0
        while ('%s.ops.%d.conv' % (prefix, n)) in self.convs or ('%s.ops.%d.conv1.conv' % (prefix, n)) in self.convs:
            n += 1
        return n

    def _build(self, B, D, H, W, train=False):
        dev, td, dt = self.device, self.tdtype, self.dt
        assert D % 16 == 0 and H % 16 == 0 and W % 16 == 0, 'spatial dims must be multiples of max_stride=16'
        split = self.split
        if split and train:
            raise RuntimeError("seg3d_b200: mode 'fp32x' is an inference mode (train in 'bf16' or 'fp32')")
        if self.wide and train:
            raise RuntimeError('seg3d_b200: training supports up to 16 classes (this net has %d); nets with up to %d classes '
                               'run inference only' % (self.out_channels, WIDE_MAX_CLASSES))
        cm = 2 if split else 1          # split mode: every activation row is [hi(C) | lo(C)]
        dims = [(D >> l, H >> l, W >> l) for l in range(5)]
        vox = [d[0] * d[1] * d[2] for d in dims]

        def buf(l, C):
            return torch.empty((B, vox[l], C * cm), dtype=td, device=dev)

        def V(b, off, ld, C):           # channel window of an activation buffer (ld = logical channel count of the buffer)
            return _View(b, off, ld * cm, C, sample=b.shape[1] * b.shape[2])

        ws = {}
        # input block as a TMA-fed Toeplitz GEMM (csrc/conv_tc_cin1t.cu): the single-channel input lives in a row-padded
        # layout [B][D][H][W + CIN1_PAD] whose padding columns stay zero (written once here, never by the gather)
        c_in = self.convs['in_block.conv']
        cin1_t = (c_in.cin1_tc and W % 8 == 0 and dt in (lib.F16, lib.BF16)
                  and os.environ.get('SEG3D_CIN1_TOEPLITZ', '1') != '0')
        ws['x_pad'] = cin1_t
        if cin1_t:
            ws['x_in'] = torch.zeros((B, D * H, W + lib.CIN1_PAD), dtype=td, device=dev)
        else:
            ws['x_in'] = torch.empty((B, vox[0], self.in_channels), dtype=torch.float32 if split else td, device=dev)
        ws['raw'] = torch.empty((B * vox[0] * 32,), dtype=torch.float32 if split else td, device=dev)
        ws['stats'] = torch.zeros((len(self.gn_names), B, 2), dtype=torch.float64, device=dev)
        ws['stats2'] = torch.zeros((B, 2), dtype=torch.float64, device=dev)
        ws['probs'] = torch.empty((B, self.out_channels, D, H, W), dtype=torch.float32, device=dev)
        widths = [32, 64, 128, 256, 256]
        for l in range(5):
            C = widths[l]
            ws['cat%d' % l] = buf(l, C) if l < 4 else None
            ws['A%d' % l] = buf(l, C) if l >= 1 else None       # down-path rblock input
            ws['T%da' % l], ws['T%db' % l] = buf(l, C), buf(l, C)
            ws['U%d' % l] = buf(l, C)                            # rblock result (up path; level 4: down_256 output)
            ws['M%da' % l], ws['M%db' % l] = buf(l, C // 4), buf(l, C // 4)   # bottleneck mids (VBNet)
        # ops: callables op(b0, nb) that launch one kernel on samples [b0, b0 + nb) of the batch; levels[i] = pyramid level
        # of op i's OUTPUT (the schedule runs the shallow levels in L2-sized sub-batches, see _schedule)
        ops, meta, units, levels = [], [], [], []
        ws['meta'], ws['units'], ws['dims'], ws['vox'], ws['B'], ws['levels'] = meta, units, dims, vox, B, levels
        ws['train'] = train
        st = lib.stream_ptr
        raw = ws['raw']

        def stats_ptr(name, b0):
            return lib.ptr(ws['stats'][self.gn_index[name]], 2 * b0)

        def add(fn, level):
            ops.append(fn)
            levels.append(level)

        def conv(name, x, xdims, y, stats_name, lout, gnin=None):
            c = self.convs[name]
            assert c.cin == x.C and c.cout == y.C, (name, c.cin, x.C, c.cout, y.C)
            if gnin is not None:       # the first gnin['nch'] input channels are a raw conv result: GroupNorm + ReLU formed on load
                gg = self.gns[gnin['gn']]
                add(lambda b0, nb: lib.call('seg3d_conv3d_k3_gnin_fwd', dt, x.at(b0), x.ld, c.cin, gnin['nch'], stats_ptr(gnin['gn'], b0),
                                            lib.ptr(gg.gamma), lib.ptr(gg.beta), GN_EPS, lib.ptr(c.w), lib.ptr(c.bias), y.at(b0), y.ld,
                                            c.cout, nb, xdims[0], xdims[1], xdims[2], stats_ptr(stats_name, b0) if stats_name else None,
                                            st()), lout)
            elif split and c.impl == lib.IMPL_TCGEN05:       # x: [hi | lo] f16 rows, y: fp32 raw
                add(lambda b0, nb: lib.call('seg3d_conv3d_split_fwd', c.mode, x.at(b0), x.ld, x.ld // 2, c.cin, lib.ptr(c.w),
                                            lib.ptr(c.bias), y.at(b0), y.ld, c.cout, nb, xdims[0], xdims[1], xdims[2],
                                            stats_ptr(stats_name, b0) if stats_name else None, st()), lout)
            elif split:                                    # input block: fp32 in, fp32 weights, fp32 out on the CUDA cores
                assert x.buf.dtype == torch.float32 and y.buf.dtype == torch.float32
                add(lambda b0, nb: lib.call('seg3d_conv3d_fwd', c.mode, lib.F32, lib.IMPL_SIMT, x.at(b0), x.ld, c.cin, lib.ptr(c.w),
                                            lib.ptr(c.bias), y.at(b0), y.ld, c.cout, nb, xdims[0], xdims[1], xdims[2],
                                            stats_ptr(stats_name, b0) if stats_name else None, st()), lout)
            else:
                add(lambda b0, nb: lib.call('seg3d_conv3d_fwd', c.mode, dt, c.call_impl, x.at(b0), x.ld, c.cin, lib.ptr(c.w),
                                            lib.ptr(c.bias), y.at(b0), y.ld, c.cout, nb, xdims[0], xdims[1], xdims[2],
                                            stats_ptr(stats_name, b0) if stats_name else None, st()), lout)
            nv_in = B * xdims[0] * xdims[1] * xdims[2]
            taps = {lib.CONV_K3: 27, lib.CONV_K2S2: 1, lib.CONV_T2S2: 8, lib.CONV_K1: 1}[c.mode]   # MACs per INPUT voxel / (cin*cout)
            nv_out = nv_in // 8 if c.mode == lib.CONV_K2S2 else (nv_in * 8 if c.mode == lib.CONV_T2S2 else nv_in)
            esz = 4 if dt == lib.F32 else 2
            kind = ('conv_tc' if c.impl == lib.IMPL_TCGEN05 else 'conv_simt') + '_' + \
                {lib.CONV_K3: 'k3', lib.CONV_K2S2: 'k2s2', lib.CONV_T2S2: 't2s2', lib.CONV_K1: 'k1'}[c.mode]
            if c.cin1_tc and xdims[2] % 8 == 0:
                kind = 'conv_tc_cin1'
            meta.append({'name': name, 'kind': kind,
                         'flops': 2.0 * nv_in * taps * c.cin * c.cout,
                         'bytes': esz * (nv_in * c.cin + nv_out * c.cout) + c.w.numel() * c.w.element_size()})

        def gn(name, y, out, nvox, relu, res, lout):
            g = self.gns[name]
            if split:
                add(lambda b0, nb: lib.call('seg3d_gn_apply_split', y.at(b0), y.ld, y.C, stats_ptr(name, b0), lib.ptr(g.gamma),
                                            lib.ptr(g.beta), GN_EPS, res.at(b0) if res is not None else None,
                                            res.ld if res is not None else 0, res.ld // 2 if res is not None else 0,
                                            out.at(b0), out.ld, out.ld // 2, 1 if relu else 0, nb, nvox, st()), lout)
            else:
                add(lambda b0, nb: lib.call('seg3d_gn_apply', dt, y.at(b0), y.ld, y.C, stats_ptr(name, b0), lib.ptr(g.gamma),
                                            lib.ptr(g.beta), GN_EPS, res.at(b0) if res is not None else None,
                                            res.ld if res is not None else 0, out.at(b0), out.ld, 1 if relu else 0, nb, nvox, st()),
                    lout)
            esz = 4 if dt == lib.F32 else 2
            meta.append({'name': name, 'kind': 'gn_apply', 'flops': 0.0,
                         'bytes': esz * B * nvox * y.C * (3 if res is not None else 2)})

        def rawview(C, l=0):
            if train:       # training keeps every pre-GroupNorm tensor for the backward pass
                return _View(torch.empty((B, vox[l], C), dtype=td, device=dev), 0, C, C, sample=vox[l] * C)
            return _View(raw, 0, C, C, sample=vox[l] * C, scratch=True)   # split mode: the raw scratch is fp32, one value per channel

        def tmpbuf(l, C, key):
            if train:
                return _View(torch.empty((B, vox[l], C), dtype=td, device=dev), 0, C, C, sample=vox[l] * C)
            return V(ws[key], 0, C, C)

        def conv_gn_twice(cname, gname, x, xdims, out, nvox_out, lout):
            """HBM-bound stride-2 / transposed conv: run it twice (statistics, then GroupNorm + ReLU in the epilogue)
            instead of storing the raw result and streaming it through seg3d_gn_apply"""
            c, g = self.convs[cname], self.gns[gname]
            esz = 2
            nv_in = B * xdims[0] * xdims[1] * xdims[2]
            taps = 1 if c.mode == lib.CONV_K2S2 else 8
            kind = 'conv_tc_' + ('k2s2' if c.mode == lib.CONV_K2S2 else 't2s2')
            for ps in (0, 1):
                add(lambda b0, nb, ps=ps: lib.call('seg3d_conv3d_gn_relu_fwd', c.mode, dt, ps, x.at(b0), x.ld, c.cin, lib.ptr(c.w),
                                                   lib.ptr(c.bias), out.at(b0), out.ld, c.cout, nb, xdims[0], xdims[1], xdims[2],
                                                   stats_ptr(gname, b0), lib.ptr(g.gamma), lib.ptr(g.beta), GN_EPS, st()), lout)
                meta.append({'name': cname + ('.stats' if ps == 0 else '.gn_relu'), 'kind': kind,
                             'flops': 2.0 * nv_in * taps * c.cin * c.cout if ps == 1 else 0.0,
                             'bytes': esz * (nv_in * c.cin + (B * nvox_out * c.cout if ps == 1 else 0)) + c.w.numel() * 2})

        # measured on B200: the stride-2 convs are epilogue-bound, not HBM-bound, so running them twice costs more than the
        # GroupNorm pass it saves (1535 vs 1640 Mvox/s); kept behind SEG3D_FUSE_S2=1
        fuse_s2_env = os.environ.get('SEG3D_FUSE_S2', '0')         # '1': every stride-2 conv; 'up': the transposed convs only
        fuse_s2 = (not train) and dt != lib.F32 and not split and fuse_s2_env in ('1', 'up')

        def unit(cname, gname, x, lin, lout, out, res=None, defer_gn=False, gnin=None):
            """conv -> GroupNorm -> (+res) -> ReLU with the conv reading level `lin` and writing level `lout`"""
            c = self.convs[cname]
            C = c.cout
            if defer_gn:        # the consumer applies GroupNorm + residual + ReLU itself (seg3d_conv3d_k3_narrow_gn_fwd)
                rv = rawview(C, lout)
                conv(cname, x, dims[lin], rv, gname, lout, gnin=gnin)
                ws['deferred'] = {'raw': rv, 'res': res, 'gn': gname, 'res_gnin': gnin}
                units.append({'conv': cname, 'gn': gname, 'x': x, 'lin': lin, 'lout': lout, 'raw': rv, 'out': out, 'res': res})
                return
            if (fuse_s2 and res is None and c.impl == lib.IMPL_TCGEN05 and out.ld % 8 == 0
                    and c.mode in ((lib.CONV_T2S2,) if fuse_s2_env == 'up' else (lib.CONV_K2S2, lib.CONV_T2S2))):
                conv_gn_twice(cname, gname, x, dims[lin], out, vox[lout], lout)
                units.append({'conv': cname, 'gn': gname, 'x': x, 'lin': lin, 'lout': lout, 'raw': None, 'out': out, 'res': res})
                return
            rv = rawview(C, lout)
            conv(cname, x, dims[lin], rv, gname, lout)
            gn(gname, rv, out, vox[lout], True, res, lout)
            units.append({'conv': cname, 'gn': gname, 'x': x, 'lin': lin, 'lout': lout, 'raw': rv, 'out': out, 'res': res})

        def conv_gn(cname, gname, x, l, out, relu, res=None, defer_gn=False, gnin=None):
            assert relu
            assert gnin is None or defer_gn
            unit(cname, gname, x, l, l, out, res, defer_gn, gnin)

        def rblock(prefix, X, l, dest, defer_last=False, gnin=None):
            n = self._rblock_len(prefix)
            C = X.C
            cur = X
            for i in range(n):
                last = i == n - 1
                out = dest if last else tmpbuf(l, C, 'T%d%s' % (l, 'ab'[i % 2]))
                op = '%s.ops.%d' % (prefix, i)
                if (op + '.conv') in self.convs:
                    conv_gn(op + '.conv', op + '.gn', cur, l, out, relu=True, res=X if last else None,
                            defer_gn=defer_last and last, gnin=gnin if (n == 1 and defer_last) else None)
                else:
                    m1 = tmpbuf(l, C // 4, 'M%da' % l)
                    m2 = tmpbuf(l, C // 4, 'M%db' % l)
                    conv_gn(op + '.conv1.conv', op + '.conv1.gn', cur, l, m1, relu=True)
                    conv_gn(op + '.conv2.conv', op + '.conv2.gn', m1, l, m2, relu=True)
                    conv_gn(op + '.conv3.conv', op + '.conv3.gn', m2, l, out, relu=True, res=X if last else None)
                cur = out
            # relu(X + ops(X)): the last apply carries relu=True with the residual (residual_block3.py:24,46);
            # for i < n-1 relu=True is ConvGnRelu3's own activation.

        # the network's last GroupNorm + residual + ReLU (up_32.rblock) has a single consumer, out_block.conv1: form it in
        # that kernel's shared memory instead of streaming it through HBM
        c1_ = self.convs['out_block.conv1']
        fuse_tail = (not train and not split and c1_.fold and c1_.impl == lib.IMPL_TCGEN05 and c1_.cin == 32 and W % 8 == 0
                     and ('up_32.rblock.ops.%d.conv' % (self._rblock_len('up_32.rblock') - 1)) in self.convs
                     and os.environ.get('SEG3D_TAIL_F32', '1') != '0' and os.environ.get('SEG3D_FUSE_TAIL', '1') != '0')

        cu_ = self.convs.get('up_32.rblock.ops.0.conv')
        fuse_up = (fuse_tail and self._rblock_len('up_32.rblock') == 1 and cu_ is not None and cu_.impl == lib.IMPL_TCGEN05
                   and cu_.cin == 32 and cu_.cout == 32 and self.convs['up_32.up_conv'].impl == lib.IMPL_TCGEN05
                   and os.environ.get('SEG3D_TC_ZMARCH', '1') != '0' and os.environ.get('SEG3D_FUSE_UP', '1') != '0')

        # in_block -> second half of cat0
        x_in = _View(ws['x_in'], 0, self.in_channels, self.in_channels, sample=vox[0] * self.in_channels)
        skip = [V(ws['cat%d' % l], widths[l] // 2, widths[l], widths[l] // 2) for l in range(4)]
        if cin1_t:
            # run the layer twice (its input is 1/16 of its output): GroupNorm sums only, then conv + GroupNorm + ReLU in the
            # epilogue - the raw tensor and the GroupNorm-apply pass of vnet_inblock.py:13-14 never touch HBM.
            # SEG3D_FUSE_IN=0: one raw pass + seg3d_gn_apply
            g_in = self.gns['in_block.gn']
            xp_sample = D * H * (W + lib.CIN1_PAD)
            xpad = _View(ws['x_in'], 0, 1, 1, sample=xp_sample)

            def cin1(epi, out):
                return lambda b0, nb: lib.call('seg3d_conv3d_cin1_fwd', dt, epi, xpad.at(b0), W + lib.CIN1_PAD, lib.ptr(c_in.w),
                                               lib.ptr(c_in.bias), out.at(b0) if out is not None else None,
                                               out.ld if out is not None else 0, nb, D, H, W, stats_ptr('in_block.gn', b0),
                                               lib.ptr(g_in.gamma), lib.ptr(g_in.beta), GN_EPS, st())
            flops = 2.0 * B * vox[0] * 27 * 16
            if not train and os.environ.get('SEG3D_FUSE_IN', '1') != '0':
                add(cin1(1, None), 0)
                meta.append({'name': 'in_block.conv.stats', 'kind': 'conv_tc_cin1', 'flops': flops, 'bytes': 2 * B * vox[0]})
                add(cin1(2, skip[0]), 0)
                meta.append({'name': 'in_block.conv.gn_relu', 'kind': 'conv_tc_cin1', 'flops': flops, 'bytes': 2 * B * vox[0] * 17})
                units.append({'conv': 'in_block.conv', 'gn': 'in_block.gn', 'x': x_in, 'lin': 0, 'lout': 0, 'raw': None,
                              'out': skip[0], 'res': None})
            else:
                rv = rawview(16, 0)
                add(cin1(0, rv), 0)
                meta.append({'name': 'in_block.conv', 'kind': 'conv_tc_cin1', 'flops': flops, 'bytes': 2 * B * vox[0] * 17})
                gn('in_block.gn', rv, skip[0], vox[0], True, None, 0)
                # training keeps the raw tensor; 'xpad': the weight gradient reads the same padded input (seg3d_conv3d_cin1_wgrad)
                units.append({'conv': 'in_block.conv', 'gn': 'in_block.gn', 'x': x_in, 'lin': 0, 'lout': 0, 'raw': rv,
                              'out': skip[0], 'res': None, 'xpad': xpad})
        else:
            conv_gn('in_block.conv', 'in_block.gn', x_in, 0, skip[0], relu=True)
        # down path
        src = skip[0]
        for l, name in ((1, 'down_32'), (2, 'down_64'), (3, 'down_128'), (4, 'down_256')):
            C = widths[l] // 2 if l < 4 else 256
            A = V(ws['A%d' % l], 0, C, C)
            unit(name + '.down_conv', name + '.down_gn', src, l - 1, l, A)
            dest = skip[l] if l < 4 else V(ws['U4'], 0, 256, 256)
            rblock(name + '.rblock', A, l, dest)
            src = dest
        # up path
        for l, name in ((3, 'up_256'), (2, 'up_128'), (1, 'up_64'), (0, 'up_32')):
            C = widths[l]
            up = V(ws['cat%d' % l], 0, C, C // 2)
            gnin = None
            if l == 0 and fuse_up:
                # the transposed convolution leaves its RAW result in the lower half of the concat buffer; both readers of that
                # half (the residual block's convolution and the residual input of the fused out-block convolution) apply
                # GroupNorm + ReLU on load, so up_32.up_gn's apply pass (vnet_upblock.py:19) never touches HBM
                conv(name + '.up_conv', src, dims[l + 1], up, name + '.up_gn', l)
                gnin = {'gn': name + '.up_gn', 'nch': C // 2}
                units.append({'conv': name + '.up_conv', 'gn': name + '.up_gn', 'x': src, 'lin': l + 1, 'lout': l, 'raw': up,
                              'out': up, 'res': None})
            else:
                unit(name + '.up_conv', name + '.up_gn', src, l + 1, l, up)
            cat = V(ws['cat%d' % l], 0, C, C)
            dest = V(ws['U%d' % l], 0, C, C)
            rblock(name + '.rblock', cat, l, dest, defer_last=(l == 0 and fuse_tail), gnin=gnin)
            src = dest
        # out block: conv1 -> raw, then the fused tail
        nc = self.out_channels
        c1 = self.convs['out_block.conv1']
        ncp = c1.cout                                      # = nc, or 16 when padded for the tensor-core path
        # conv1's raw output feeds GN1 -> 1x1x1 conv -> GN2 -> softmax directly: its storage rounding would dominate
        # the probability error, so the tensor-core path stores it in fp32 (64 B/voxel instead of 32)
        tail_f32 = (c1.impl == lib.IMPL_TCGEN05 and src.C in (16, 32, 64) and W % 8 == 0 and not train and not split
                    and os.environ.get('SEG3D_TAIL_F32', '1') != '0')
        tail_dt = lib.F32 if (tail_f32 or split) else dt
        if self.wide:
            # raw conv1 result in fp32 rows of pitch wide_cp (a multiple of 4 floats, as the tail's TMA needs) in every mode:
            # the z-march kernel up to 64 padded channels (32 in fp32x), the generic tensor-core kernel above, SIMT in fp32
            ncp = self.wide_cp
            rv1 = _View(torch.empty((B, vox[0], ncp), dtype=torch.float32, device=dev), 0, ncp, c1.cout, sample=vox[0] * ncp)
            if dt == lib.F32 or split:
                conv('out_block.conv1', src, dims[0], rv1, 'out_block.gn1', 0)
            else:
                add(lambda b0, nb: lib.call('seg3d_conv3d_fwd', c1.mode, dt | lib.OUT_F32, c1.impl, src.at(b0), src.ld, c1.cin,
                                            lib.ptr(c1.w), lib.ptr(c1.bias), rv1.at(b0), rv1.ld, c1.cout, nb, dims[0][0], dims[0][1],
                                            dims[0][2], stats_ptr('out_block.gn1', b0), st()), 0)
                meta.append({'name': 'out_block.conv1', 'kind': 'conv_tc_k3', 'flops': 2.0 * B * vox[0] * 27 * c1.cin * c1.cout,
                             'bytes': 2 * B * vox[0] * c1.cin + 4 * B * vox[0] * c1.cout + c1.w.numel() * 2})
        elif tail_f32 and c1.fold:
            # nine in-plane taps folded into the GEMM N dimension (csrc/conv_tc_narrow.cu), fp32 result
            ncp = nc
            rv1 = _View(torch.empty((B, vox[0], nc), dtype=torch.float32, device=dev), 0, nc, nc, sample=vox[0] * nc)
            dfr = ws.get('deferred')
            if dfr is not None:
                g0 = self.gns[dfr['gn']]
                draw, dres, dgn, rgn = dfr['raw'], dfr['res'], dfr['gn'], dfr.get('res_gnin')
                if rgn is not None:       # the residual's lower half is still raw (fuse_up above)
                    gr = self.gns[rgn['gn']]
                    add(lambda b0, nb: lib.call('seg3d_conv3d_k3_narrow_gn2_fwd', dt, draw.at(b0), draw.ld, dres.at(b0), dres.ld, c1.cin,
                                                stats_ptr(dgn, b0), lib.ptr(g0.gamma), lib.ptr(g0.beta), GN_EPS,
                                                rgn['nch'], stats_ptr(rgn['gn'], b0), lib.ptr(gr.gamma), lib.ptr(gr.beta),
                                                lib.ptr(c1.w_fold), lib.ptr(c1.bias), rv1.at(b0), nc, nb, dims[0][0], dims[0][1],
                                                dims[0][2], stats_ptr('out_block.gn1', b0), st()), 0)
                else:
                    add(lambda b0, nb: lib.call('seg3d_conv3d_k3_narrow_gn_fwd', dt, draw.at(b0), draw.ld, dres.at(b0), dres.ld, c1.cin,
                                                stats_ptr(dgn, b0), lib.ptr(g0.gamma), lib.ptr(g0.beta), GN_EPS,
                                                lib.ptr(c1.w_fold), lib.ptr(c1.bias), rv1.at(b0), nc, nb, dims[0][0], dims[0][1], dims[0][2],
                                                stats_ptr('out_block.gn1', b0), st()), 0)
                rd = 2 * (2 * B * vox[0] * c1.cin)
            else:
                add(lambda b0, nb: lib.call('seg3d_conv3d_k3_narrow_fwd', dt, src.at(b0), src.ld, c1.cin, lib.ptr(c1.w_fold),
                                            lib.ptr(c1.bias), rv1.at(b0), nc, nb, dims[0][0], dims[0][1], dims[0][2],
                                            stats_ptr('out_block.gn1', b0), st()), 0)
                rd = 2 * B * vox[0] * c1.cin
            meta.append({'name': 'out_block.conv1', 'kind': 'conv_tc_narrow', 'flops': 2.0 * B * vox[0] * 27 * c1.cin * nc,
                         'bytes': rd + 4 * B * vox[0] * nc + c1.w_fold.numel() * 2})
        elif split and c1.fold and c1.impl == lib.IMPL_TCGEN05 and src.C == 32 and src.off == 0 and src.ld == 64 and W % 8 == 0:
            # strict mode: the same folded kernel on split operands (rows [hi(32) | lo(32)]), fp32 result
            ncp = nc
            rv1 = _View(torch.empty((B, vox[0], nc), dtype=torch.float32, device=dev), 0, nc, nc, sample=vox[0] * nc)
            add(lambda b0, nb: lib.call('seg3d_conv3d_k3_narrow_split_fwd', src.at(b0), src.ld, c1.cin, lib.ptr(c1.w_fold),
                                        lib.ptr(c1.bias), rv1.at(b0), nc, nb, dims[0][0], dims[0][1], dims[0][2],
                                        stats_ptr('out_block.gn1', b0), st()), 0)
            meta.append({'name': 'out_block.conv1', 'kind': 'conv_tc_narrow', 'flops': 2.0 * B * vox[0] * 27 * c1.cin * nc,
                         'bytes': 2 * 2 * B * vox[0] * c1.cin + 4 * B * vox[0] * nc + c1.w_fold.numel() * 2})
        elif tail_f32:
            ncp = nc                                       # the fp32 store keeps only the real channels
            rv1 = _View(torch.empty((B, vox[0], nc), dtype=torch.float32, device=dev), 0, nc, nc, sample=vox[0] * nc)
            add(lambda b0, nb: lib.call('seg3d_conv3d_fwd', c1.mode, dt | lib.OUT_F32, c1.impl, src.at(b0), src.ld, c1.cin, lib.ptr(c1.w),
                                        lib.ptr(c1.bias), rv1.at(b0), rv1.ld, c1.cout, nb, dims[0][0], dims[0][1], dims[0][2],
                                        stats_ptr('out_block.gn1', b0), st()), 0)
            meta.append({'name': 'out_block.conv1', 'kind': 'conv_tc_k3', 'flops': 2.0 * B * vox[0] * 27 * c1.cin * c1.cout,
                         'bytes': 2 * B * vox[0] * c1.cin + 4 * B * vox[0] * nc + c1.w.numel() * 2})
        else:
            rv1 = rawview(ncp, 0)           # the two tail launches of a sub-batch read it before the next sub-batch rewrites it
            conv('out_block.conv1', src, dims[0], rv1, 'out_block.gn1', 0)
        ws['tail'] = {'x': src, 'raw': rv1, 'ncp': ncp}
        g1, g2 = self.gns['out_block.gn1'], self.gns['out_block.gn2']
        probs = ws['probs']
        psample = self.out_channels * vox[0]

        def tail_stats(b0, nb):
            lib.call('seg3d_outblock_tail_stats', tail_dt, rv1.at(b0), ncp, nc, stats_ptr('out_block.gn1', b0), lib.ptr(g1.gamma),
                     lib.ptr(g1.beta), lib.ptr(self.w2), lib.ptr(self.b2), GN_EPS, lib.ptr(ws['stats2'], 2 * b0), nb, vox[0], st())

        def tail_probs(b0, nb):
            lib.call('seg3d_outblock_tail_probs', tail_dt, rv1.at(b0), ncp, nc, stats_ptr('out_block.gn1', b0), lib.ptr(g1.gamma),
                     lib.ptr(g1.beta), lib.ptr(self.w2), lib.ptr(self.b2), lib.ptr(ws['stats2'], 2 * b0), lib.ptr(g2.gamma),
                     lib.ptr(g2.beta), GN_EPS, lib.ptr(probs, b0 * psample), nb, vox[0], st())

        if self.wide:
            def tail_wide(ps):
                return lambda b0, nb: lib.call('seg3d_outblock_tail_wide', ps, rv1.at(b0), rv1.ld, nc, stats_ptr('out_block.gn1', b0),
                                               lib.ptr(g1.gamma), lib.ptr(g1.beta), lib.ptr(self.w2), lib.ptr(self.b2), GN_EPS,
                                               lib.ptr(ws['stats2'], 2 * b0), lib.ptr(g2.gamma), lib.ptr(g2.beta),
                                               lib.ptr(probs, b0 * psample), nb, vox[0], st())
            add(tail_wide(0), 0)
            add(tail_wide(1), 0)
            # per voxel: 3 * Cp / 16 MMAs of K = 16 on Cp columns; pass 0 reads the raw row, pass 1 reads it and writes C probs
            flops = 2.0 * 3 * B * vox[0] * ncp * ncp
            meta.append({'name': 'out_block.tail_stats', 'kind': 'tail_wide', 'flops': flops, 'bytes': 4 * B * vox[0] * ncp})
            meta.append({'name': 'out_block.tail_probs', 'kind': 'tail_wide', 'flops': flops,
                         'bytes': 4 * B * vox[0] * ncp + 4 * B * vox[0] * nc})
            ws['schedule'] = self._schedule(B, levels, vox, train)
            return ws, ops
        add(tail_stats, 0)
        add(tail_probs, 0)
        esz = 4 if dt == lib.F32 else 2
        esz = 4 if (tail_f32 or split) else esz
        meta.append({'name': 'out_block.tail_stats', 'kind': 'tail', 'flops': 0.0, 'bytes': esz * B * vox[0] * ncp})
        meta.append({'name': 'out_block.tail_probs', 'kind': 'tail', 'flops': 0.0, 'bytes': esz * B * vox[0] * ncp + 4 * B * vox[0] * nc})
        ws['schedule'] = self._schedule(B, levels, vox, train)
        return ws, ops

    def _schedule(self, B, levels, vox, train):
        """[(first op, last op + 1, sub-batch)]: the order in which run() issues the launches.
        The levels 0 and 1 of the pyramid are HBM-bound (GroupNorm applies, stride-2 / transposed convs, the input block and the
        narrow out-block conv move whole 16-32-channel tensors and do little math); their tensors are 28-57 MB per 96^3
        patch, so a batch of 20 streams every one of them through HBM between producer and consumer.  GroupNorm is per
        sample and every op is a batched launch, so each maximal run of consecutive level <= 1 ops is issued in sub-batches
        of a few patches: the raw conv output a GroupNorm apply reads, and the activation the next conv reads, are then
        still in the 126 MB L2, and the raw scratch is re-written in place by the next sub-batch before it is ever evicted.
        The deep levels (small tensors, tensor-bound, better at a large batch) run once over the whole batch.
        SEG3D_SUBBATCH_MB = L2 budget for one sub-batch's level-0 working set (0 = no sub-batching)."""
        budget = float(os.environ.get('SEG3D_SUBBATCH_MB', '0')) * 1e6
        n = len(levels)
        if train or budget <= 0 or B <= 1:
            return [(0, n, B)]
        per_sample = vox[0] * 32 * (4 if self.dt == lib.F32 else 2) * (2 if self.split else 1)    # one 32-channel level-0 tensor
        sb = int(max(1, min(B, budget // per_sample)))
        sched, i = [], 0
        while i < n:
            j = i
            shallow = levels[i] <= 1
            while j < n and (levels[j] <= 1) == shallow:
                j += 1
            sched.append((i, j, sb if shallow else B))
            i = j
        return sched

    def plan(self, B, D, H, W, train=False):
        """(workspaces, launch list) for one input shape.  The cache is a small LRU (SEG3D_PLAN_CACHE shapes, default 4):
        whole-volume forwards (partition_type 'DISABLE') have a different shape per case, and an unbounded cache would
        keep ~430 B/voxel of workspace alive for every case ever seen."""
        key = (B, D, H, W, train)
        hit = self._plans.pop(key, None)
        if hit is None:
            limit = max(1, int(os.environ.get('SEG3D_PLAN_CACHE', '4')))
            while len(self._plans) >= limit:
                self._plans.pop(next(iter(self._plans)))          # least recently used: dicts keep insertion order
            hit = self._build(B, D, H, W, train)
        self._plans[key] = hit
        return hit

    def load_input(self, ws, x):
        """x: [B,Cin,D,H,W] float32 CUDA tensor -> NDHWC storage dtype."""
        B = x.shape[0]
        if ws.get('x_pad'):
            D, H, W = x.shape[2:]
            ws['x_in'].view(B, D, H, W + lib.CIN1_PAD)[..., lib.CIN1_LEFT:lib.CIN1_LEFT + W].copy_(x[:, 0])
        elif self.in_channels == 1:
            ws['x_in'].view(-1).copy_(x.reshape(-1))
        else:
            ws['x_in'].copy_(x.reshape(B, self.in_channels, -1).permute(0, 2, 1))

    def _run_eager(self, ws, ops):
        ws['stats'].zero_()
        ws['stats2'].zero_()
        B = ws['B']
        for i0, i1, sb in ws['schedule']:
            for b0 in range(0, B, sb):
                nb = min(sb, B - b0)
                for op in ops[i0:i1]:
                    op(b0, nb)

    def launches(self, ws):
        """kernel launches of one forward under the plan's schedule"""
        B = ws['B']
        return sum((i1 - i0) * ((B + sb - 1) // sb) for i0, i1, sb in ws['schedule'])

    def run(self, ws, ops):
        """One forward over the plan's workspaces.  With SEG3D_GRAPH=1 an inference plan is captured into a CUDA graph after
        one eager run (all buffers, packed weights and tensor maps are fixed per plan) and replayed afterwards: the launches of
        a forward become one, which matters for small patch batches and for sub-batched schedules."""
        if self.use_graph and not ws.get('train', False):
            g = ws.get('graph')
            if g is None:
                self._run_eager(ws, ops)              # lazy one-time setup inside the library happens outside the capture
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._run_eager(ws, ops)
                ws['graph'] = g
            g.replay()
        else:
            self._run_eager(ws, ops)
        self.launches_per_forward = self.launches(ws)
        return ws['probs']

    def run_profiled(self, ws, ops):
        """Same as run() with a CUDA-event pair around every launch (current stream).  Returns
        [(meta dict, milliseconds)], the launches of one op (sub-batches) summed - used by bench.py for the per-kernel
        roofline table."""
        ws['stats'].zero_()
        ws['stats2'].zero_()
        B = ws['B']
        evs = [[] for _ in ops]
        for i0, i1, sb in ws['schedule']:
            for b0 in range(0, B, sb):
                nb = min(sb, B - b0)
                for i in range(i0, i1):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    ops[i](b0, nb)
                    b.record()
                    evs[i].append((a, b))
        torch.cuda.synchronize()
        return [(m, sum(a.elapsed_time(b) for a, b in e)) for m, e in zip(ws['meta'], evs)]

    def forward(self, x):
        """probabilities [B,C,D,H,W] float32 (a view of the plan's output buffer; clone to keep)."""
        _require_cuda(x.device, 'seg3d_b200: input must be a CUDA tensor (no CPU fallback)')
        B, Cin, D, H, W = x.shape
        assert Cin == self.in_channels
        ws, ops = self.plan(B, D, H, W)
        self.load_input(ws, x.float())
        return self.run(ws, ops)


DEFAULT_TC_MODES = (lib.CONV_K3, lib.CONV_K2S2, lib.CONV_T2S2)
WIDE_MAX_CLASSES = 127
