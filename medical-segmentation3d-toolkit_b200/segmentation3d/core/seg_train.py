"""Training engine (drop-in for reference segmentation3d/core/seg_train.py:22-153).

Same config file, folder layout, logging and checkpoint cadence.  The step itself
(zero_grad -> net(crops) -> loss -> backward -> Adam, :119-127) runs the network and the loss on the C-ABI
kernels.  Multi-GPU is one process per GPU (launch with torchrun): per-rank batch = train.batchsize, gradients are
averaged with a bucketed NCCL all-reduce (segmentation3d/_b200/dist.py) in place of nn.DataParallel (:77); rank 0
logs and writes checkpoints, with the `module.` key prefix the reference's GPU loader expects.
"""
import importlib
import os
import shutil
import time

import numpy as np
import torch
import torch.optim as optim
from torch.utils.data import DataLoader

from segmentation3d._b200 import dist as D
from segmentation3d.dataloader.dataset import SegmentationDataset
from segmentation3d.dataloader.sampler import EpochConcateDistributedSampler, EpochConcateSampler
from segmentation3d.loss.cross_entropy_loss import CrossEntropyLoss
from segmentation3d.loss.focal_loss import FocalLoss
from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
from segmentation3d.utils.file_io import load_config, setup_logger
from segmentation3d.utils.image_tools import save_intermediate_results
from segmentation3d.utils.model_io import load_checkpoint, save_checkpoint


class _ModulePrefixed(object):
    """state_dict() with the DataParallel 'module.' prefix, so checkpoints load in the reference GPU path."""

    def __init__(self, net):
        self.net = net

    def state_dict(self):
        return {'module.' + k: v for k, v in self.net.state_dict().items()}


def make_loss(train_cfg, use_gpu=True):
    name = train_cfg.loss.name
    if name == 'Focal':
        return FocalLoss(class_num=train_cfg.dataset.num_classes, alpha=train_cfg.loss.obj_weight,
                         gamma=train_cfg.loss.focal_gamma, use_gpu=use_gpu)
    if name == 'Dice':
        return MultiDiceLoss(weights=train_cfg.loss.obj_weight, num_class=train_cfg.dataset.num_classes, use_gpu=use_gpu)
    if name == 'CE':
        return CrossEntropyLoss()
    raise ValueError('Unknown loss function')


def make_optimizer(net, lr, betas=(0.9, 0.999)):
    """The reference's optim.Adam(net.parameters(), lr, betas) (core/seg_train.py:83): a torch.optim.Adam subclass - same
    state-dict layout, same update rule - whose step() is one C-ABI launch over all parameters (_b200/optim.py)."""
    from segmentation3d._b200.optim import FlatAdam
    root = getattr(net, 'module', net)
    on_step = getattr(root, 'mark_weights_changed', None)
    if on_step is None:
        # a network assembled from the standalone modules re-packs a convolution's weights when the parameter's version
        # counter moves (blocks.packed_conv); the Adam kernel writes the parameters behind torch's back, so move it here
        params = list(net.parameters())

        def on_step():
            torch.autograd.graph.increment_version(params)
    return FlatAdam(net.parameters(), lr=lr, betas=betas, on_step=on_step)


def train_step(net, opt, loss_func, crops, masks, params=None, return_outputs=False):
    """core/seg_train.py:119-127 for one batch already on the device; returns the loss tensor (and, on request, the
    probabilities the loss was computed from)."""
    opt.zero_grad()
    outputs = net(crops)
    loss = loss_func(outputs, masks)
    loss.backward()
    plan = getattr(getattr(net, 'module', net), '_plan', None)
    if not getattr(plan, 'grads_reduced_in_backward', False):      # else: already averaged, overlapped with the backward pass
        D.allreduce_mean_grads(params if params is not None else list(net.parameters()))
    opt.step()
    return (loss, outputs.detach()) if return_outputs else loss


def train(train_config_file):
    assert os.path.isfile(train_config_file), 'Config not found: {}'.format(train_config_file)
    train_cfg = load_config(train_config_file)
    if train_cfg.general.num_gpus <= 0:
        raise RuntimeError('segmentation3d (B200 build) has no CPU training path: set general.num_gpus >= 1')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if train_cfg.general.num_gpus > 1 and world == 1:
        raise RuntimeError('multi-GPU training runs one process per GPU: launch with '
                           '`python -m torch.distributed.run --nproc-per-node %d -m segmentation3d.seg_train -i <cfg>`'
                           % train_cfg.general.num_gpus)
    torch.cuda.set_device(local)
    if world > 1 and not torch.distributed.is_initialized():
        torch.distributed.init_process_group('nccl', device_id=torch.device('cuda:%d' % local))

    model_folder = os.path.join(train_cfg.general.save_dir, train_cfg.general.model_scale)
    if rank == 0:
        if os.path.isdir(model_folder):
            if train_cfg.general.resume_epoch < 0:
                shutil.rmtree(model_folder)
                os.makedirs(model_folder)
        else:
            os.makedirs(model_folder)
        shutil.copy(train_config_file, os.path.join(model_folder, 'train_config.py'))
        infer_cfg = os.path.join(os.path.dirname(os.path.dirname(__file__)), 'config', 'infer_config.py')
        shutil.copy(infer_cfg, os.path.join(train_cfg.general.save_dir, 'infer_config.py'))
    if world > 1:
        torch.distributed.barrier()
    logger = setup_logger(os.path.join(model_folder, 'train_log.txt' if rank == 0 else 'train_log_rank%d.txt' % rank), 'seg3d')

    np.random.seed(train_cfg.general.seed + rank)
    torch.manual_seed(train_cfg.general.seed)
    torch.cuda.manual_seed(train_cfg.general.seed)

    dataset = SegmentationDataset(
        imlist_file=train_cfg.general.imseg_list, num_classes=train_cfg.dataset.num_classes, spacing=train_cfg.dataset.spacing,
        crop_size=train_cfg.dataset.crop_size, sampling_method=train_cfg.dataset.sampling_method,
        random_translation=train_cfg.dataset.random_translation, random_scale=train_cfg.dataset.random_scale,
        interpolation=train_cfg.dataset.interpolation, crop_normalizers=train_cfg.dataset.crop_normalizers)
    if world > 1:
        sampler = EpochConcateDistributedSampler(dataset, train_cfg.train.epochs, 0, rank=rank, world_size=world,
                                                 seed=train_cfg.general.seed)
    else:
        sampler = EpochConcateSampler(dataset, train_cfg.train.epochs)
    if os.environ.get('SEG3D_DEVICE_CROPS', '0') == '1':
        # opt-in: volumes resident in HBM, crops drawn by seg3d_crop_resample (dataloader/device_loader.py)
        from segmentation3d.dataloader.device_loader import DeviceCropLoader
        data_loader = DeviceCropLoader(dataset, sampler, train_cfg.train.batchsize, device='cuda:%d' % local)
    else:
        data_loader = DataLoader(dataset, sampler=sampler, batch_size=train_cfg.train.batchsize,
                                 num_workers=train_cfg.train.num_threads, pin_memory=True)

    net_module = importlib.import_module('segmentation3d.network.' + train_cfg.net.name)
    net = net_module.SegmentationNet(dataset.num_modality(), train_cfg.dataset.num_classes)
    max_stride = net.max_stride()
    net_module.parameters_kaiming_init(net)
    net = net.cuda()
    D.broadcast_params(net)
    assert np.all(np.array(train_cfg.dataset.crop_size) % max_stride == 0), 'crop size not divisible by max stride'

    opt = make_optimizer(net, train_cfg.train.lr, train_cfg.train.betas)
    if train_cfg.general.resume_epoch >= 0:
        last_save_epoch, batch_start = load_checkpoint(train_cfg.general.resume_epoch, _StripPrefixLoader(net), opt, model_folder)
    else:
        last_save_epoch, batch_start = 0, 0
    loss_func = make_loss(train_cfg, True)

    writer = None
    if rank == 0:
        try:
            from torch.utils.tensorboard import SummaryWriter
            writer = SummaryWriter(os.path.join(model_folder, 'tensorboard'))
        except Exception:
            writer = None

    batch_idx = batch_start
    params = list(net.parameters())
    global_batch = train_cfg.train.batchsize * world
    for crops, masks, frames, filenames in data_loader:
        begin_t = time.time()
        crops, masks = crops.cuda(non_blocking=True), masks.cuda(non_blocking=True)
        if 'debug' in train_cfg and train_cfg.debug.get('save_inputs', False):       # core/seg_train.py:130-133
            train_loss, outputs = train_step(net, opt, loss_func, crops, masks, params, return_outputs=True)
            save_intermediate_results(list(range(crops.size(0))), crops.cpu(), masks.cpu(), outputs.cpu(), frames, filenames,
                                      os.path.join(model_folder, 'batch_{}'.format(batch_idx - batch_start)))
        else:
            train_loss = train_step(net, opt, loss_func, crops, masks, params)
        epoch_idx = batch_idx * global_batch // len(dataset)
        batch_idx += 1
        loss_value = train_loss.item()
        sample_duration = (time.time() - begin_t) / train_cfg.train.batchsize
        logger.info('epoch: {}, batch: {}, train_loss: {:.4f}, time: {:.4f} s/vol'.format(epoch_idx, batch_idx, loss_value, sample_duration))
        if rank == 0 and epoch_idx != 0 and epoch_idx % train_cfg.train.save_epochs == 0 and last_save_epoch != epoch_idx:
            save_checkpoint(_ModulePrefixed(net), opt, epoch_idx, batch_idx, train_cfg, max_stride, dataset.num_modality())
            last_save_epoch = epoch_idx
        if writer is not None:
            writer.add_scalar('Train/Loss', loss_value, batch_idx)
    if writer is not None:
        writer.close()


class _StripPrefixLoader(object):
    """load_state_dict that accepts checkpoints with or without the 'module.' prefix."""

    def __init__(self, net):
        self.net = net

    def load_state_dict(self, sd):
        if any(k.startswith('module.') for k in sd):
            sd = {k[7:]: v for k, v in sd.items()}
        return self.net.load_state_dict(sd)
