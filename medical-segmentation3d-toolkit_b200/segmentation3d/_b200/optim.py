"""Adam on the C-ABI kernel (reference core/seg_train.py:83 `optim.Adam(net.parameters(), lr=..., betas=...)`, :127 `opt.step()`).

`FlatAdam` IS a torch.optim.Adam - same constructor, param_groups, state_dict()/load_state_dict() (so `optimizer.pth` of
utils/model_io.py keeps its layout: per parameter `step`, `exp_avg`, `exp_avg_sq`) - whose step() is ONE seg3d_adam_step
launch: the parameters of its group are re-homed, once, as views of one flat fp32 buffer, so are the moments, and the
gradients arrive as views of one flat buffer in the same layout from the network's backward pass (autograd.py::_param_grads).
Gradients that arrive any other way (a user-made .grad) are copied into a flat scratch first.  As in torch.optim.Adam, a
parameter whose .grad is None is skipped: its value, moments and its own `step` stay as they are.  Parameters then can
have different step counts, and such steps go through seg3d_adam_step_ranges (one range per run of parameters with a
gradient and the same step count); a step in which every parameter has a gradient and all counts agree stays one
seg3d_adam_step launch.  Configurations the kernel does not implement (amsgrad, maximize, several groups, sparse / non-fp32 / non-CUDA parameters) take torch's own step().
"""
import torch

from . import lib
from .packing import flat_layout


class FlatAdam(torch.optim.Adam):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, on_step=None):
        super().__init__(list(params), lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self._on_step = on_step
        self._flat = None               # (param flat, exp_avg flat, exp_avg_sq flat, offsets, total, per-parameter step tensors)
        self._counts = None             # the step counts as host ints (what step() decides on), kept equal to the tensors
        self._gscratch = None

    # ---------------------------------------------------------------------------------------------------------------
    def _kernel_ok(self):
        if len(self.param_groups) != 1:
            return False
        g = self.param_groups[0]
        if g.get('amsgrad') or g.get('maximize') or g.get('capturable') or g.get('differentiable'):
            return False
        ps = g['params']
        return len(ps) > 0 and all(self._on_device(p) and p.dtype == torch.float32 and p.device == ps[0].device and not p.is_sparse
                                   for p in ps)

    @staticmethod
    def _on_device(p):          # a function of its own so the CPU wiring tests (kernels emulated) can lift it; the package never does
        return p.is_cuda

    def _adopt(self):
        """re-home parameters and moments as views of flat buffers (existing values and state are carried over)"""
        ps = self.param_groups[0]['params']
        named = [(str(i), p) for i, p in enumerate(ps)]
        offsets, total = flat_layout(named)
        dev = ps[0].device
        flat = torch.zeros((total,), dtype=torch.float32, device=dev)
        m = torch.zeros_like(flat)
        v = torch.zeros_like(flat)
        steps = []
        for (key, p) in named:
            o, n = offsets[key], p.numel()
            flat[o:o + n].copy_(p.data.reshape(-1))
            p.data = flat[o:o + n].view(p.shape)
            st = self.state[p]
            if 'exp_avg' in st:
                m[o:o + n].copy_(st['exp_avg'].reshape(-1))
                v[o:o + n].copy_(st['exp_avg_sq'].reshape(-1))
            st['step'] = torch.tensor(float(st['step']) if 'step' in st else 0.0, dtype=torch.float32)
            steps.append(st['step'])
            st['exp_avg'] = m[o:o + n].view(p.shape)
            st['exp_avg_sq'] = v[o:o + n].view(p.shape)
        self._flat = (flat, m, v, [offsets[k] for k, _ in named], total, steps)
        self._counts = [int(float(st)) for st in steps]

    def _adopted(self):
        if self._flat is None:
            return False
        flat, m, v, offs, total, steps = self._flat
        base, mb = flat.data_ptr(), m.data_ptr()
        for p, o, step in zip(self.param_groups[0]['params'], offs, steps):
            st = self.state.get(p)
            if p.data_ptr() != base + 4 * o or st is None or st.get('step') is not step or st['exp_avg'].data_ptr() != mb + 4 * o:
                return False
        return True

    def _flat_grads(self):
        """a flat gradient tensor laid out like the parameters: the buffer the backward pass handed out when every .grad that
        is not None is still a view of it, else a scratch the gradients are copied into (the slots of parameters without a
        gradient are not read)"""
        flat, _, _, offs, total, _ = self._flat
        ps = self.param_groups[0]['params']
        k0 = next(i for i, p in enumerate(ps) if p.grad is not None)
        g0 = ps[k0].grad
        if g0.dtype == torch.float32:
            store, s0 = g0.untyped_storage(), g0.storage_offset() - offs[k0]
            if (s0 >= 0 and store.nbytes() >= 4 * (s0 + total) and (store.data_ptr() + 4 * s0) % 16 == 0 and
                    all(p.grad is None or (p.grad.dtype == torch.float32 and p.grad.is_contiguous() and
                                           p.grad.untyped_storage().data_ptr() == store.data_ptr() and
                                           p.grad.storage_offset() == s0 + o)
                        for p, o in zip(ps, offs))):
                return torch.empty((0,), dtype=torch.float32, device=g0.device).set_(store, s0, (total,), (1,))
        if self._gscratch is None or self._gscratch.numel() != total:
            self._gscratch = torch.zeros((total,), dtype=torch.float32, device=flat.device)
        for p, o in zip(ps, offs):
            if p.grad is not None:
                self._gscratch[o:o + p.numel()].copy_(p.grad.reshape(-1))
        return self._gscratch

    def _ranges(self, active):
        """seg3d_adam_range table of the parameters with a gradient: runs of neighbours with the same step count merged
        (the 16-byte alignment gaps between them hold zeros in every flat buffer, which the update leaves at zero)"""
        offs = self._flat[3]
        ps = self.param_groups[0]['params']
        runs = []
        for p, o, s, a in zip(ps, offs, self._counts, active):
            if not a:
                continue
            if runs and runs[-1][2] == s and runs[-1][0] + (runs[-1][1] + 3) // 4 * 4 == o:
                runs[-1][1] = o + p.numel() - runs[-1][0]
            else:
                runs.append([o, p.numel(), s])
        table = (lib.AdamRange * len(runs))()
        for e, (o, n, s) in zip(table, runs):
            e.offset, e.n, e.step = o, n, s
        return table

    @torch.no_grad()
    def step(self, closure=None):
        if not self._kernel_ok():
            self._flat = None
            return super().step(closure)
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if not self._adopted():
            self._adopt()
        flat, m, v, offs, total, steps = self._flat
        g = self.param_groups[0]
        active = [p.grad is not None for p in g['params']]
        if not any(active):
            return loss
        gflat = self._flat_grads()
        self.used_flat_grads = gflat is not self._gscratch
        every = all(active)
        torch._foreach_add_(steps if every else [st for st, a in zip(steps, active) if a], 1)      # one call, not one per tensor
        self._counts = [c + 1 for c in self._counts] if every else [c + a for c, a in zip(self._counts, active)]
        b1, b2 = g['betas']
        hyper = (float(g['lr']), float(b1), float(b2), float(g['eps']), float(g['weight_decay']))
        with torch.cuda.device(flat.device):
            if every and len(set(self._counts)) == 1:
                lib.call('seg3d_adam_step', lib.ptr(flat), lib.ptr(gflat), lib.ptr(m), lib.ptr(v), total, *hyper,
                         self._counts[0], lib.stream_ptr())
            else:
                table = self._ranges(active)
                lib.call('seg3d_adam_step_ranges', lib.ptr(flat), lib.ptr(gflat), lib.ptr(m), lib.ptr(v), table, len(table),
                         *hyper, lib.stream_ptr())
        if self._on_step is not None:
            self._on_step()
        return loss
