"""Headline benchmark: sliding-window VNet inference on a synthetic 512x512x400 CT volume, plus the training step.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

A "step" is one pass of the hot path over one volume: crop+normalise 180 patches of 96^3
(partition_size = partition_stride = 96 mm at 1 mm spacing), VNet forward, overlap blend,
normalise by the overlap count, first-argmax mask.  Metric (BASELINE.json): Mvoxels/s =
volume voxels / time.

  N = 1   `value`: the volume already in HBM (BASELINE configs[1]); `e2e`: the reference-facing call
          (segmentation3d.core.seg_infer.segmentation_volume_host) with a HOST volume - pinned H2D copy in, int8 mask D2H
          out - inside the timed region.
  N > 1   ONE volume, its patches dealt over the N ranks in contiguous z runs (`--shard patches`, the default for N > 1:
          "scaling": "strong"); the exchange step (max all-reduce of the int8 label mask when patches do not overlap,
          otherwise reduce-scatter of probability slabs + all-gather of the mask) is INSIDE the timed region.  The
          case-sharded figure (every rank its own volume, no data-path collective, BASELINE configs[4] style) is the
          `weak` sub-record.  `--shard cases` makes that one the headline instead.

Every line also carries
  `train`   BASELINE configs[2] (the second half of BASELINE.json's metric): VNet, 96^3 crops, batch 8 per GPU, MultiDiceLoss,
            Adam, data parallel over the same N ranks with the gradient all-reduce overlapped with the backward pass;
            patches/s, ms/step, roofline (3 x forward flops x batch / time against the sustained tensor peak), and at N = 1
            the CPU training step beside it;
  `parity`  (N = 1) the GPU result of this very run against the CPU reference path on the patches the `cpu_baseline` leg
            computed - both arms read the identical host array.

`--impl reference` times the reference's own CPU path (the oracle port of core/seg_infer.segmentation_volume: two forwards
per patch, numpy blend with the reference's whole-volume copies; validated at 0.992x the unmodified reference's time by
tests/golden/time_reference_cpu.py) on ALL host cores (torch's thread count is set explicitly: torchrun exports
OMP_NUM_THREADS=1), on a bounded sample of patches of the same workload; its line carries the CPU training step as `train`.
`--task train` prints the training record as a line of its own.
`--dump-outputs DIR` writes what the last timed step returned (see write_outputs) for comparing two builds output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True       # the benchmark may run from a read-only tree and writes nothing into it

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'medical-segmentation3d-toolkit_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


import numpy as np   # noqa: E402
import torch         # noqa: E402

def init_nccl(dev):
    """init_process_group with NCCL's start-up banner ("NCCL version ..." is printf'ed to stdout by the first communicator) sent to
    stderr: stdout carries exactly ONE JSON line."""
    import torch.distributed as dist
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group('nccl', device_id=torch.device(dev))
        dist.barrier()                       # the communicator (and its banner) exists before stdout is restored
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    return dist


METRIC = 'sliding-window infer Mvoxels/s (512x512x400 CT, VNet, 96^3 patches)'  # BASELINE.json headline (configs[1]); main() renames it for --arch vbnet
TRAIN_METRIC = 'train patches/s (VNet, 96^3 patches, batch %d/GPU, Dice, Adam)'
NORMALIZER = {'type': 0, 'mean': 0.0, 'stddev': 1000.0, 'clip': True}
DTYPE_NAME = {'fp16': 'f16', 'bf16': 'bf16', 'fp32': 'f32', 'fp32x': 'f16x2'}
VNET_GFLOP_PER_PATCH = 180.80          # SURVEY A.2: 2*MACs of all convolutions of one 96^3 VNet(1,2) forward


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def use_all_host_cores():
    """The CPU arms use every core the process may run on, whatever OMP_NUM_THREADS the launcher exported."""
    n = host_cores()
    torch.set_num_threads(n)
    return n


def synth_ct(size_xyz, seed):
    """Seeded CT-like volume [z,y,x] float32 in HU on the HOST: smooth low-frequency field + noise.  Both arms (GPU and
    CPU reference) read this one array."""
    g = torch.Generator(device='cpu').manual_seed(seed)
    X, Y, Z = size_xyz
    lo = torch.randn((1, 1, max(2, Z // 32), max(2, Y // 32), max(2, X // 32)), generator=g)
    field = torch.nn.functional.interpolate(lo, size=(Z, Y, X), mode='trilinear', align_corners=False)[0, 0]
    noise = torch.randn((Z, Y, X), generator=g)
    vol = field.mul_(600.0).add_(noise.mul_(60.0)).sub_(200.0).clamp_(-1000.0, 2000.0)
    return vol.float().contiguous()


def make_net(mode, arch='vnet', classes=2):
    import importlib
    mod = importlib.import_module('segmentation3d.network.' + arch)
    torch.manual_seed(0)
    net = mod.SegmentationNet(1, classes)
    mod.parameters_kaiming_init(net)
    net.b200_mode = mode
    return net


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [v.strip() for v in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {'sm_mhz': med, 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': len(sm)}


DUMP_INFER_BYTES = 48 << 20   # sampled probabilities + mask of the last inference step
DUMP_PARAMS = 1 << 20         # sampled parameter values after the last training step (4 MB): the dump stays under 64 MB


def flat_sample(n, k, device):
    """Flat indices into an output of n elements: all of them when n <= k, otherwise about k sorted distinct ones drawn
    from a fixed seed, so every run and every build samples the same elements."""
    if n <= k:
        return torch.arange(n, device=device)
    return torch.from_numpy(np.unique(np.random.default_rng(0).integers(0, n, k))).to(device)


def sample_infer_outputs(probs, mask):
    """(probabilities [C, ...] fp32, label mask int8) of one sliding-window pass -> float32 host arrays [C, k] and [k]."""
    C = probs.shape[0]
    k = DUMP_INFER_BYTES // (4 * (C + 1))
    p, m = probs.reshape(C, -1), mask.reshape(-1)
    return {'infer_probs': p[:, flat_sample(p.shape[1], k, p.device)].float().cpu().numpy(),
            'infer_mask': m[flat_sample(m.numel(), k, m.device)].float().cpu().numpy()}


def write_outputs(path, arrays):
    """DIR/<name>.npy per array: infer_probs / infer_mask (a fixed sample of the voxels of the last timed inference
    step), train_loss and train_params (the loss and a fixed sample of the flattened parameters after the last timed
    training step)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + '.npy'), a)


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        d = json.load(open(path))
        return d.get('hbm_gbs', 6536.0), d.get('bf16_tflops', 1641.1), d.get('bf16_tflops_sustained', 1382.6), 'measured'
    return 6650.0, 1590.0, 1400.0, 'fallback'


# ---- CPU arms (the only place bench.py executes oracle/) ----------------------------------------------------------
def cpu_reference_sample(vol_np, size_xyz, patch, stride, n_patches, arch='vnet', classes=2, keep=False):
    """Reference CPU path (oracle port) on the first n_patches of the workload.
    Returns dict(value Mvox/s, seconds, cores, total patches[, probs, mask, starts of the sampled patches])."""
    from oracle import init as oinit
    from oracle import sliding_window as osw
    cores = use_all_host_cores()
    sd = oinit.init_state_dict(arch, 1, classes, 0)
    total = len(osw.partition_grid(size_xyz, [1, 1, 1], [0, 0, 0], list(size_xyz), [patch] * 3, [stride] * 3, 16)[0])
    n_patches = min(n_patches, total)
    t0 = time.time()
    probs, mask, starts, ends = osw.segmentation_volume(sd, vol_np, [1.0, 1.0, 1.0], NORMALIZER, 'SIZE', [patch] * 3, [stride] * 3, 16,
                                                        double_forward=True, faithful_copies=True, max_patches=n_patches)
    dt = time.time() - t0
    vox = float(size_xyz[0]) * size_xyz[1] * size_xyz[2] * n_patches / total
    out = {'value': vox / dt / 1e6, 'seconds': dt, 'cores': cores, 'total': total, 'patches': n_patches}
    if keep:
        out.update(probs=probs, mask=mask, starts=starts[:n_patches], ends=ends[:n_patches])
    return out


def cpu_train_sample(patch, batch, steps=1):
    """Reference CPU training step (core/seg_train.py:119-127 through the oracle's autograd program: forward, Dice loss,
    backward, Adam) on `batch` crops of patch^3.  Returns (patches/s, seconds, cores)."""
    from oracle import init as oinit
    from oracle import loss as oloss
    from oracle import net as onet
    cores = use_all_host_cores()
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-4, betas=(0.9, 0.999))
    g = torch.Generator().manual_seed(0)
    crops = torch.randn((batch, 1, patch, patch, patch), generator=g)
    masks = torch.randint(0, 2, (batch, 1, patch, patch, patch), generator=g).float()
    t0 = time.time()
    for _ in range(steps):
        opt.zero_grad()
        loss = oloss.multi_dice_loss(onet.forward_with_grad(params, crops), masks, [0.5, 0.5])
        loss.backward()
        opt.step()
    dt = time.time() - t0
    return batch * steps / dt, dt, cores


def cpu_train_record(args):
    v, dt, cores = cpu_train_sample(args.patch, 1)
    return {'value': v, 'unit': 'patches/s', 'cores': cores, 'kind': 'port',
            'sample': '1 training step on 1 crop of %d^3 (forward, Dice, backward, Adam; fp32), %.1f s' % (args.patch, dt)}


def train_config(args, world, mode):
    return {'workload': 'VNet(1,2) training step, crops [%d,1,%d^3] per GPU, MultiDiceLoss, Adam lr 1e-4 (BASELINE configs[2])'
                        % (args.train_batch, args.patch), 'mode': mode, 'parallelism': 'dp%d' % world}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    size = [int(v) for v in args.volume.split(',')]
    if args.task == 'train':
        vals = [cpu_train_sample(args.patch, 1) for _ in range(args.warmup + args.steps)][args.warmup:]
        value, dt, cores = float(np.mean([v[0] for v in vals])), float(np.mean([v[1] for v in vals])), vals[0][2]
        sample = '1 training step on 1 crop of %d^3 per timed step (forward, Dice, backward, Adam; fp32)' % args.patch
        print(json.dumps({
            'impl': 'reference', 'metric': TRAIN_METRIC % args.train_batch,
            'value': value, 'unit': 'patches/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': train_config(args, args.gpus, 'fp32'),
            'cpu_baseline': {'value': value, 'unit': 'patches/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': 'patches/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}))
        return
    vol_np = synth_ct(size, 1234).numpy()
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_reference_sample(vol_np, size, args.patch, args.stride, args.ref_patches, args.arch, args.classes)
        if i >= args.warmup:
            vals.append(r)
    value = float(np.mean([r['value'] for r in vals]))
    ms = float(np.mean([r['seconds'] for r in vals])) * 1e3
    spread = (max(r['value'] for r in vals) - min(r['value'] for r in vals)) / value if len(vals) > 1 else 0.0
    sample = ('%d of %d patches per timed step (x2 forwards each, as core/seg_infer.py:230-234) through the reference loop incl. '
              'whole-volume numpy copies; extrapolated linearly in the patch count (every patch costs the same two forwards and the same '
              'copies); spread over the %d timed steps %.1f %%' % (vals[0]['patches'], vals[0]['total'], len(vals), 100 * spread))
    line = {
        'impl': 'reference', 'metric': metric_name(args), 'value': value, 'unit': 'Mvoxels/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True,
        'scaling': 'strong' if (args.gpus > 1 and args.shard != 'cases') else 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, size, args.gpus),
        'cpu_baseline': {'value': value, 'unit': 'Mvoxels/s', 'cores': vals[0]['cores'], 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'Mvoxels/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    if not args.no_train:
        t = cpu_train_record(args)
        line['train'] = {'metric': TRAIN_METRIC % args.train_batch, 'value': t['value'], 'unit': 'patches/s', 'dtype': 'f32',
                         'cpu_baseline': t, 'config': train_config(args, args.gpus, 'fp32')}
    print(json.dumps(line))


def metric_name(args):
    return METRIC if args.arch == 'vnet' else METRIC.replace('VNet', 'VBNet C=%d' % args.classes)


def workload_config(args, size, world):
    shard = args.shard if world > 1 else None
    return {'workload': '%s(1,%d) random-init sliding-window inference, volume %dx%dx%d @1mm, partition_size=%d mm, '
                        'partition_stride=%d mm (BASELINE configs[%d])' % ({'vnet': 'VNet', 'vbnet': 'VBNet'}[args.arch], args.classes,
                                                                           size[0], size[1], size[2], args.patch, args.stride,
                                                                           1 if args.arch == 'vnet' else 3),
            'patch_batch': args.batch, 'mode': args.mode, 'shard': shard, 'gather': args.gather if shard == 'patches' else None,
            'l2_policy': 'inputs larger than L2 (volume 419 MB + accumulators 839 MB per step)'}


# ---- training step (BASELINE configs[2]) ----------------------------------------------------------------------------
def measure_train(args, dist, rank, world, dev, cpu_leg=True):
    """VNet, 96^3 crops, batch 8/GPU, MultiDiceLoss, Adam(lr 1e-4); data parallel over the ranks of `dist` (None: one GPU).
    The timed region is the reference's step window (core/seg_train.py:119-127) on device-resident synthetic batches."""
    from segmentation3d._b200 import dist as D
    from segmentation3d.core.seg_train import make_optimizer, train_step
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    mode = args.train_mode
    net = make_net(mode).to(dev).train()
    D.broadcast_params(net)
    opt = make_optimizer(net, 1e-4, (0.9, 0.999))
    lf = MultiDiceLoss([0.5, 0.5], 2, True)
    B, P = args.train_batch, args.patch
    g = torch.Generator(device=dev).manual_seed(rank)
    crops = torch.randn((B, 1, P, P, P), generator=g, device=dev)
    masks = torch.randint(0, 2, (B, 1, P, P, P), generator=g, device=dev).float()
    params = list(net.parameters())
    warm = max(args.warmup, 3)
    for _ in range(warm):
        loss = train_step(net, opt, lf, crops, masks, params)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = train_step(net, opt, lf, crops, masks, params)
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    loss_value = float(loss.item())
    outputs = None
    if args.dump_outputs and rank == 0:
        flat = torch.cat([p.detach().reshape(-1).float() for p in params])
        outputs = {'train_loss': np.array([loss_value], np.float64),
                   'train_params': flat[flat_sample(flat.numel(), DUMP_PARAMS, flat.device)].cpu().numpy()}
        del flat
    resolved = net.resolve_mode(train=True)
    del net, opt, crops, masks
    torch.cuda.empty_cache()
    if rank != 0:
        return None, None
    _, _, tf_sust, which = peaks()
    flops = 3.0 * VNET_GFLOP_PER_PATCH * 1e9 * B * (P / 96.0) ** 3        # forward + data gradient + weight gradient, per GPU
    rec = {
        'metric': TRAIN_METRIC % B, 'value': B * world / (ms * 1e-3), 'unit': 'patches/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': warm, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
        'dtype': DTYPE_NAME[resolved], 'data': 'synthetic', 'config': train_config(args, world, resolved), 'loss': loss_value,
        'roofline': {'bound': 'tensor', 'achieved': flops / (ms * 1e-3) / 1e12, 'peak': tf_sust, 'unit': 'TFLOP/s',
                     'frac': flops / (ms * 1e-3) / 1e12 / tf_sust, 'traffic': None,
                     'algorithmic_flops_per_step_per_gpu': flops,
                     'note': 'whole step (forward, loss, backward, all-reduce, Adam): 3 x 180.8 GFLOP x batch / step time, per GPU',
                     'peak_source': which},
        'collective': None if world == 1 else 'all-reduce(sum) of the flat fp32 gradient buffer (58.3 MB), issued tail-first in '
                                              '~12 MB pieces on NCCL\'s stream while the backward pass is still running',
    }
    if cpu_leg and world == 1 and not args.no_cpu_baseline:
        rec['cpu_baseline'] = cpu_train_record(args)
    return rec, outputs


def run_train(args):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = 'cuda:%d' % local
    dist = None
    if world > 1:
        dist = init_nccl(dev)
    rec, outputs = measure_train(args, dist, rank, world, dev)
    if rank == 0:
        rec['vs_baseline'] = None
        if args.dump_outputs:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(rec))
    if dist is not None:
        dist.destroy_process_group()


# ---- inference ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--mode', default='fp16', choices=['auto', 'fp16', 'bf16', 'fp32', 'fp32x'],
                    help="fp32x = strict parity on the tensor cores (f16 hi/lo split operands, fp32 accumulate)")
    ap.add_argument('--train-mode', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--batch', type=int, default=36, help='patches per network forward (36 = one z layer of the 6x6x5 patch grid)')
    ap.add_argument('--volume', default='512,512,400')
    ap.add_argument('--patch', type=int, default=96)
    ap.add_argument('--stride', type=int, default=96)
    ap.add_argument('--shard', default=None, choices=['cases', 'patches'],
                    help="N > 1: 'patches' (default) = ONE volume, patches dealt over the ranks, exchange step timed (strong scaling); "
                         "'cases' = every rank its own volume (weak scaling)")
    ap.add_argument('--gather', default='labels', choices=['mask', 'probs', 'labels'],
                    help="--shard patches: 'labels' = local arg-max + max all-reduce of the int8 mask (non-overlapping patches; "
                         "falls back to 'mask' otherwise); 'mask' = reduce-scatter of probability slabs + all-gather of the mask; "
                         "'probs' = all-reduce of the probability maps")
    ap.add_argument('--ref-patches', type=int, default=None,
                    help='patches in the bounded CPU sample (default: 8 for the cpu_baseline leg of a GPU run, 4 per timed step of --impl reference)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-train', action='store_true', help='skip the training sub-record')
    ap.add_argument('--no-weak', action='store_true', help='N > 1: skip the case-sharded sub-record')
    ap.add_argument('--layers', action='store_true', help='print the per-kernel roofline table to stderr')
    ap.add_argument('--task', default='infer', choices=['infer', 'train'],
                    help="'train': the training record (BASELINE configs[2], patches/s) as a line of its own")
    ap.add_argument('--train-batch', type=int, default=8)
    ap.add_argument('--arch', default='vnet', choices=['vnet', 'vbnet'], help='vbnet + --classes 5 = BASELINE configs[3]')
    ap.add_argument('--classes', type=int, default=2)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned to DIR/<name>.npy (float32/float64, under 64 MB: fixed seeded '
                         'samples of the larger outputs; the inputs are the same in every run)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs records the GPU path; --impl reference has no such outputs')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.shard is None:
        args.shard = 'patches' if max(world, args.gpus if args.impl == 'reference' else 1) > 1 else 'cases'
    if args.ref_patches is None:
        args.ref_patches = 4 if args.impl == 'reference' else 8
    if args.impl == 'reference':
        return run_reference(args)
    if args.task == 'train':
        return run_train(args)

    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (the product has no CPU fallback)'
    torch.cuda.set_device(local)
    dev = 'cuda:%d' % local
    dist = None
    if world > 1:
        dist = init_nccl(dev)

    from segmentation3d._b200 import lib
    from segmentation3d.core.seg_infer import segmentation_volume_device, segmentation_volume_host, make_model
    lib.load()
    size = [int(v) for v in args.volume.split(',')]
    nvox = float(size[0]) * size[1] * size[2]
    net = make_net(args.mode, args.arch, args.classes).to(dev).eval()
    model = make_model(net, spacing=[1.0, 1.0, 1.0], normalizer=NORMALIZER)
    cfg = {'partition_type': 'SIZE', 'partition_size': [args.patch] * 3, 'partition_stride': [args.stride] * 3}
    patches = world > 1 and args.shard == 'patches'
    # the identical host array feeds the GPU arm and the CPU reference arm (one volume when patch-sharded, one per rank else)
    host_src = synth_ct(size, 1234 + (0 if (patches or world == 1) else rank))
    host_vol = torch.empty(host_src.shape, dtype=torch.float32, pin_memory=True)
    host_vol.copy_(host_src)
    vol = host_vol.to(dev)
    host_mask = torch.empty(vol.shape, dtype=torch.int8, pin_memory=True)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = model['engine'].kernel_launches
        e0.record()
        for _ in range(steps):
            out = None          # the previous step's outputs go back to the allocator before the next step allocates its own
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = model['engine'].kernel_launches - l0
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, launches, out

    def measure(shard_mode):
        shard = (rank, world) if (shard_mode == 'patches' and world > 1) else None
        ms_dev, launches, out = timed(lambda: segmentation_volume_device(model, cfg, vol, batch=args.batch, shard=shard, gather=args.gather),
                                      args.steps, max(args.warmup, 3))
        # sharded: the merged mask is reduced to rank 0, the one process that copies it out (and would write the result file)
        ms_e2e, _, _ = timed(lambda: segmentation_volume_host(model, cfg, host_vol, host_mask, batch=args.batch, shard=shard, gather=args.gather,
                                                              mask_root=0 if shard is not None else None),
                             args.steps, 3)
        units = nvox * (world if shard is None else 1)
        return {'value': units / (ms_dev * 1e-3) / 1e6, 'ms_per_step': ms_dev, 'launches': launches,
                'e2e': units / (ms_e2e * 1e-3) / 1e6, 'ms_e2e': ms_e2e}, out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    head, last = measure(args.shard)
    clocks = sampler.stop() if rank == 0 else None
    dump = sample_infer_outputs(*last) if (args.dump_outputs and rank == 0) else {}
    del last
    weak = None
    if world > 1 and args.shard == 'patches' and not args.no_weak:
        # every rank its own copy of the volume: replicas only, no collective on the data path
        weak, _ = measure('cases')

    # parity of this very run: the device result of the single-GPU pass against the CPU reference on the sampled patches
    parity, cpu = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        acc, mask = segmentation_volume_device(model, cfg, vol, batch=args.batch)
        torch.cuda.synchronize()
        r = cpu_reference_sample(host_src.numpy(), size, args.patch, args.stride, args.ref_patches, args.arch, args.classes, keep=True)
        cpu = {'value': r['value'], 'unit': 'Mvoxels/s', 'cores': r['cores'], 'kind': 'port',
               'sample': '%d of %d patches (x2 forwards, reference loop incl. whole-volume numpy copies), %.1f s; linear in the patch '
                         'count (every patch costs the same two forwards and the same copies)' % (r['patches'], r['total'], r['seconds'])}
        # compare every voxel all of whose contributing patches are in the CPU sample (clamped last boxes overlap their neighbours)
        from oracle import sliding_window as osw
        all_s, all_e = osw.partition_grid(size, [1, 1, 1], [0, 0, 0], list(size), [args.patch] * 3, [args.stride] * 3, 16)
        full = np.zeros((size[2], size[1], size[0]), np.int16)
        part = np.zeros_like(full)
        for s0, e0 in zip(all_s, all_e):
            full[s0[2]:e0[2], s0[1]:e0[1], s0[0]:e0[0]] += 1
        for s0, e0 in zip(r['starts'], r['ends']):
            part[s0[2]:e0[2], s0[1]:e0[1], s0[0]:e0[0]] += 1
        valid = (part == full) & (part > 0)
        zs = np.flatnonzero(valid.any(axis=(1, 2)))
        z0, z1 = int(zs.min()), int(zs.max()) + 1
        gp = acc[:, z0:z1].cpu().numpy()
        gm = mask[z0:z1].cpu().numpy()
        v = valid[z0:z1]
        nv = int(v.sum())
        parity = {'max_abs_dprob': float(np.abs(gp - r['probs'][:, z0:z1])[:, v].max()),
                  'label_agreement': float((gm == r['mask'][z0:z1])[v].sum()) / nv, 'voxels': nv,
                  'bars': 'reduced precision: max_abs <= 1e-2, agreement >= 0.999 (BASELINE.json north_star)',
                  'against': 'CPU reference path (oracle port, fp32) on the same host array, %d patches' % r['patches']}
        del acc, mask

    # per-kernel table from one instrumented forward of a full patch batch
    roof, shares = None, None
    if rank == 0:
        hbm, tf_burst, tf_sust, which = peaks()
        plan = net._current_plan()
        ws, ops = plan.plan(args.batch, args.patch, args.patch, args.patch)
        plan.run_profiled(ws, ops)
        prof = plan.run_profiled(ws, ops)
        kinds = {}
        for m, ms in prof:
            k = kinds.setdefault(m['kind'], {'ms': 0.0, 'flops': 0.0, 'bytes': 0.0, 'n': 0})
            k['ms'] += ms; k['flops'] += m['flops']; k['bytes'] += m['bytes']; k['n'] += 1
        tot_ms = sum(k['ms'] for k in kinds.values())
        if args.layers:
            for m, ms in prof:
                sys.stderr.write('%-34s %-14s %8.3f ms %8.1f TFLOP/s %8.1f GB/s\n' % (
                    m['name'], m['kind'], ms, m['flops'] / ms / 1e9, m['bytes'] / ms / 1e6))
            for kname, k in sorted(kinds.items(), key=lambda kv: -kv[1]['ms']):
                sys.stderr.write('KIND %-14s n=%3d %8.3f ms (%4.1f%%) %8.1f TFLOP/s %8.1f GB/s\n' % (
                    kname, k['n'], k['ms'], 100 * k['ms'] / tot_ms, k['flops'] / k['ms'] / 1e9, k['bytes'] / k['ms'] / 1e6))
        top = max(kinds.items(), key=lambda kv: kv[1]['ms'])
        tk = top[1]
        if top[0].startswith('conv_tc'):
            roof = {'bound': 'tensor', 'achieved': tk['flops'] / tk['ms'] / 1e9, 'peak': tf_sust, 'unit': 'TFLOP/s'}
        else:
            roof = {'bound': 'hbm', 'achieved': tk['bytes'] / tk['ms'] / 1e6, 'peak': hbm, 'unit': 'GB/s'}
        roof['frac'] = roof['achieved'] / roof['peak']
        # DRAM bytes per launch of this kernel class from the committed ncu --set full capture (tools/make_profiles.py),
        # scaled to this run's patch batch; null when no capture of this class exists
        roof['traffic'] = None
        for tname in ('r02_traffic.json', 'r01_traffic.json'):
            tpath = os.path.join(ROOT, 'profiles', tname)
            if os.path.isfile(tpath) and args.arch == 'vnet' and args.mode == 'fp16':
                tj = json.load(open(tpath))
                if top[0] in tj:
                    roof['traffic'] = tj[top[0]]['dram_bytes_per_launch'] * args.batch / float(tj.get('_batch', args.batch))
                    roof['traffic_source'] = tj.get('_source')
                    roof['algorithmic_bytes_per_launch'] = tk['bytes'] / tk['n']
                    break
        roof['kernel'] = top[0]
        roof['share_of_forward'] = tk['ms'] / tot_ms
        roof['peak_source'] = which + ' (MEASURED_PEAKS.json, sustained)' if which == 'measured' else which
        roof['launches_per_forward'] = tk['n']
        roof['avg_launch_ms'] = tk['ms'] / tk['n']
        shares = {k: round(v['ms'] / tot_ms, 4) for k, v in kinds.items()}
        del ws, ops

    # the training half of the metric, same ranks
    train = None
    if not args.no_train:
        del vol
        model['engine'].plan = None
        net._plans.clear()
        net._plan = None
        torch.cuda.empty_cache()
        train, train_out = measure_train(args, dist, rank, world, dev)
        if train_out:
            dump.update(train_out)

    if rank == 0:
        resolved = net.resolve_mode()
        line = {
            'metric': metric_name(args), 'value': head['value'], 'unit': 'Mvoxels/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': head['ms_per_step'], 'higher_is_better': True,
            'scaling': 'strong' if patches else 'weak', 'vs_baseline': None,
            'dtype': DTYPE_NAME[resolved], 'data': 'synthetic',
            'config': workload_config(args, size, world),
            'e2e': {'value': head['e2e'], 'unit': 'Mvoxels/s', 'ms_per_step': head['ms_e2e'],
                    'h2d_bytes_per_step': int(nvox * 4) if not patches else None, 'd2h_bytes_per_step': int(nvox)},
            'gpu_launches': head['launches'], 'clocks': clocks, 'roofline': roof, 'cpu_baseline': cpu, 'parity': parity,
            'kernel_shares': shares,
        }
        if patches:
            from segmentation3d.core.seg_infer import shard_plan
            _, _, mine, (z_lo, z_hi), disjoint = shard_plan(model, cfg, (size[2], size[1], size[0]), (0, world))
            line['e2e']['h2d_bytes_per_step'] = int((z_hi - z_lo) * size[1] * size[0] * 4)
            line['e2e']['note'] = 'per rank: only the z planes its patches read are uploaded (h2d_bytes_per_step = rank 0); the merged mask is reduced to rank 0, which copies it out'
            line['collective'] = ('max all-reduce of the int8 label mask (%d MB) after a local count-normalise + arg-max of each '
                                  'rank\'s z range (whole overlap components are dealt to one rank)' % int(nvox / 1e6)) if (args.gather == 'labels' and disjoint) else \
                ('per-class reduce-scatter of fp32 probability slabs (%d MB) + all-gather of the int8 mask' % int(nvox * 4 * args.classes / 1e6)
                 if args.gather != 'probs' else 'all-reduce of the fp32 probability maps (%d MB)' % int(nvox * 4 * args.classes / 1e6))
            line['patches_per_rank'] = len(mine)
        if weak is not None:
            line['weak'] = {'metric': metric_name(args), 'value': weak['value'], 'unit': 'Mvoxels/s', 'scaling': 'weak',
                            'ms_per_step': weak['ms_per_step'], 'e2e': {'value': weak['e2e'], 'unit': 'Mvoxels/s', 'ms_per_step': weak['ms_e2e']},
                            'config': {'shard': 'cases', 'note': 'every rank segments its own 512x512x400 volume; no data-path collective'}}
        if train is not None:
            line['train'] = train
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
