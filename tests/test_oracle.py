"""The oracle against the golden fixtures produced by the live reference (tests/golden/make_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import init as oinit
from oracle import loss as oloss
from oracle import net as onet
from oracle import sliding_window as osw
from oracle.metrics import cal_dsc

G = os.path.join(os.path.dirname(__file__), 'golden')
GOLDEN_THREADS = 8              # tests/golden/make_golden.py computes every fixture with torch.set_num_threads(8)


@pytest.fixture(autouse=True)
def golden_threads():
    """oneDNN divides a CPU convolution among the threads, and the division sets the fp32 summation order: the oracle
    reproduces the fixtures to the last bits only with the thread count that computed them, whatever the host's count."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def seeded_input(seed, shape, kind='noise'):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g)
    if kind == 'smooth':
        lo = torch.randn((shape[0], shape[1]) + tuple(max(2, s // 8) for s in shape[2:]), generator=g)
        x = torch.nn.functional.interpolate(lo, size=shape[2:], mode='trilinear', align_corners=False) * 2 + 0.3 * x
    return x


def sd_hash(sd):
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(v.detach().contiguous().numpy().tobytes())
    return h.hexdigest()


def test_schema_matches_reference():
    schema = json.load(open(os.path.join(G, 'schema.json')))
    for key, ref in schema.items():
        arch, cin, cout = key.split('_')
        mine = oinit.state_dict_schema(arch, int(cin), int(cout))
        assert [[k, list(s)] for k, s in mine] == ref
    assert sum(int(np.prod(s)) for _, s in oinit.state_dict_schema('vnet', 1, 2)) == 14563296   # SURVEY a1
    assert sum(int(np.prod(s)) for _, s in oinit.state_dict_schema('vbnet', 1, 5)) == 8666727   # SURVEY a2


def test_seeded_init_is_bit_identical_to_reference():
    hashes = json.load(open(os.path.join(G, 'weights_sha256.json')))
    for key, ref in hashes.items():
        arch, cin, cout, seed, mode = key.split('_')
        sd = oinit.init_state_dict(arch, int(cin), int(cout), int(seed[4:]), mode)
        assert sd_hash(sd) == ref, key


def test_forward_matches_reference():
    z = np.load(os.path.join(G, 'forward.npz'))
    meta = json.loads(str(z['meta']))
    for name, arch, cin, cout, wseed, aseed, iseed, shape, kind in meta:
        sd = oinit.init_state_dict(arch, cin, cout, wseed)
        if aseed is not None:
            sd = oinit.randomize_affine(sd, aseed)
        y = onet.forward(sd, seeded_input(iseed, tuple(shape), kind)).numpy()
        assert y.shape == z[name].shape
        # same ATen ops in the same order: bit-equal in practice, allow 1 ulp-ish slack
        assert np.abs(y - z[name]).max() <= 1e-6, name


def test_module_prefix_is_stripped():
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    x = seeded_input(3, (1, 1, 16, 16, 16))
    a = onet.forward(sd, x)
    b = onet.forward({'module.' + k: v for k, v in sd.items()}, x)
    assert torch.equal(a, b)


def test_partition_grid_bit_exact():
    cases = json.load(open(os.path.join(G, 'grids.json')))
    assert len(cases) >= 10
    for c in cases:
        bs = list(c['bbox_start']) if c['bbox_start'] is not None else [0, 0, 0]
        be = list(c['bbox_end']) if c['bbox_end'] is not None else list(c['size'])
        s, e = osw.partition_grid(c['size'], c['spacing'], bs, be, list(c['partition_size']),
                                  list(c['partition_stride']), 16)
        assert s == c['starts'] and e == c['ends']
        assert bs == c['bbox_start_after'] and be == c['bbox_end_after']   # in-place mutation, image_tools.py:184-187
    # SURVEY A.3 table
    n = {(tuple(c['size']), c['partition_stride'][0]): c['n'] for c in cases if c['bbox_start'] is None}
    assert n[((512, 512, 400), 96)] == 180 and n[((512, 512, 400), 48)] == 800
    assert n[((256, 256, 256), 96)] == 27 and n[((256, 256, 256), 48)] == 125


def test_losses_match_reference():
    z = np.load(os.path.join(G, 'loss.npz'))
    for c in (2, 5):
        k = 'c%d_' % c
        probs, target, w = torch.from_numpy(z[k + 'probs']), torch.from_numpy(z[k + 'target']), z[k + 'weights'].tolist()
        p = probs.clone().requires_grad_(True)
        l = oloss.multi_dice_loss(p, target, w)
        l.backward()
        assert abs(float(l) - float(z[k + 'dice'])) <= 1e-7
        assert np.abs(p.grad.numpy() - z[k + 'dice_grad']).max() <= 1e-9
        p = probs.clone().requires_grad_(True)
        l = oloss.focal_loss(p, target, c, alpha=w, gamma=2, size_average=True)
        l.backward()
        assert abs(float(l) - float(z[k + 'focal'])) <= 1e-7
        assert np.abs(p.grad.numpy() - z[k + 'focal_grad']).max() <= 1e-9
        p = probs.clone().requires_grad_(True)
        l = oloss.focal_loss(p, target, c, alpha=None, gamma=0, size_average=False)
        l.backward()
        assert abs(float(l) - float(z[k + 'focal_g0_sum'])) <= 1e-3 * abs(float(z[k + 'focal_g0_sum'])) * 1e-3 + 1e-4
        assert np.abs(p.grad.numpy() - z[k + 'focal_g0_sum_grad']).max() <= 1e-6
        # closed form used by the fused CUDA reduction (SURVEY 3.4)
        terms = oloss.multi_dice_terms(probs, target)
        wn = np.array(w) / np.sum(w)
        per = 1.0 - (2 * terms[:, :, 0] + 1e-6) / (terms[:, :, 1] + terms[:, :, 2] + 1e-6)
        closed = float((per.mean(0).numpy() * wn).sum())
        assert abs(closed - float(z[k + 'dice'])) <= 1e-6
    l = oloss.binary_dice_loss(torch.from_numpy(z['bin_probs']), torch.from_numpy(z['bin_target']))
    assert abs(float(l) - float(z['bin_dice'])) <= 1e-7


def test_sliding_window_matches_reference():
    z = np.load(os.path.join(G, 'sliding_window.npz'))
    meta = json.loads(str(z['meta']))
    for name, arch, cout, wseed, aseed, size, psize, pstride, norm, vseed, scale in meta:
        sd = oinit.init_state_dict(arch, 1, cout, wseed)
        if aseed is not None:
            sd = oinit.randomize_affine(sd, aseed)
        vol = (seeded_input(vseed, (1, 1, size[2], size[1], size[0]), 'smooth')[0, 0].numpy() * scale).astype(np.float32)
        if norm[0] == 'fixed':
            nd = {'type': 0, 'mean': norm[1], 'stddev': norm[2], 'clip': norm[3]}
        else:
            nd = {'type': 1, 'clip_sigma': norm[1]}
        probs, mask, starts, ends = osw.segmentation_volume(sd, vol, [1.0, 1.0, 1.0], nd, 'SIZE', psize, pstride, 16)
        assert np.abs(probs - z[name + '_probs']).max() <= 1e-6, name
        assert (mask == z[name + '_mask']).mean() >= 0.99999, name
        # single forward == double forward (SURVEY D5), and no-copy accumulate == faithful accumulate
        if name == 'sw_vnet_adaptive':
            p1, m1, _, _ = osw.segmentation_volume(sd, vol, [1.0, 1.0, 1.0], nd, 'SIZE', psize, pstride, 16,
                                                   double_forward=False, faithful_copies=False)
            assert np.array_equal(p1, probs) and np.array_equal(m1, mask)
        cnt = osw.overlap_count_axes(size, starts, ends)
        assert cnt.min() >= 1


def test_sliding_window_64_patches_matches_reference():
    """the 64^3-patch goldens (probabilities committed on every 2nd voxel per axis, masks in full)"""
    z = np.load(os.path.join(G, 'sliding_window_64.npz'))
    for name, arch, cout, wseed, aseed, size, psize, pstride, norm, vseed, scale in json.loads(str(z['meta'])):
        if name != 'sw64_vnet_tiled':       # one case keeps the CPU suite short; the other is covered by the GPU test's fp32x arm
            continue
        sd = oinit.init_state_dict(arch, 1, cout, wseed)
        vol = (seeded_input(vseed, (1, 1, size[2], size[1], size[0]), 'smooth')[0, 0].numpy() * scale).astype(np.float32)
        nd = {'type': 0, 'mean': norm[1], 'stddev': norm[2], 'clip': norm[3]} if norm[0] == 'fixed' else {'type': 1, 'clip_sigma': norm[1]}
        probs, mask, _, _ = osw.segmentation_volume(sd, vol, [1.0, 1.0, 1.0], nd, 'SIZE', psize, pstride, 16,
                                                    double_forward=False, faithful_copies=False)
        assert np.abs(probs[:, ::2, ::2, ::2] - z[name + '_probs']).max() <= 1e-6, name
        assert (mask == z[name + '_mask']).mean() >= 0.99999, name


def test_argmax_ties_pick_lowest_class():
    p = np.zeros((3, 2, 2, 2), np.float32)
    p[:] = 1.0 / 3
    p[2, 0, 0, 0] = 0.5
    m = osw.argmax_first(p)
    assert m.dtype == np.int8 and m[0, 0, 0] == 2 and m[1, 1, 1] == 0


def test_cal_dsc():
    a = np.zeros((4, 4, 4), np.int8)
    b = np.zeros((4, 4, 4), np.int8)
    a[:2] = 1
    b[1:3] = 1
    assert cal_dsc(a, b, 1, 1) == (0.5, 'TP')
    assert cal_dsc(a, b, 2, 1) == (1.0, 'TN')
    assert cal_dsc(a, np.zeros_like(a), 1, 1) == (0.0, 'FN')


def test_resample_out_size_rounding():
    assert osw.resample_out_size([512, 512, 400], [1, 1, 1], [1, 1, 1], 16) == [512, 512, 400]
    assert osw.resample_out_size([300, 300, 200], [0.5, 0.5, 1.0], [0.4, 0.4, 0.4], 16) == [384, 384, 512]


def test_oracle_resample_restatement_known_answers():
    """oracle/resample.py (ITK Resample semantics, parity unpinned): hand-checked 1-D cases embedded in 3-D."""
    from oracle import resample as orz
    line = np.array([0.0, 10.0, 20.0, 40.0], dtype=np.float32)
    src = np.broadcast_to(line, (2, 3, 4)).copy()
    # same spacing, same size: identity
    assert np.array_equal(orz.resample_grid(src, [1, 1, 1], [4, 3, 2], [1, 1, 1], 'LINEAR'), src)
    # x spacing 1 -> 0.5: c = 0, .5, 1, ..., 3.5 ; c < 3.5 is inside, c = 3.5 gets the default value
    out = orz.resample_grid(src, [1, 1, 1], [8, 3, 2], [0.5, 1, 1], 'LINEAR', default_value=-7.0)
    assert np.allclose(out[0, 0], [0, 5, 10, 15, 20, 30, 40, -7.0])
    # between the last sample and the buffer edge the upper neighbour is clamped (c = 3.25 -> 40)
    out = orz.resample_grid(src, [1, 1, 1], [14, 3, 2], [0.25, 1, 1], 'LINEAR', default_value=-7.0)
    assert out[0, 0, 13] == 40.0 and out[1, 2, 12] == 40.0 and out[0, 0, 1] == 2.5
    # nearest: floor(c + 0.5)
    out = orz.resample_grid(src, [1, 1, 1], [8, 3, 2], [0.5, 1, 1], 'NN', default_value=-7.0)
    assert np.array_equal(out[0, 0], np.array([0, 10, 10, 20, 20, 40, 40, -7.0], dtype=np.float32))
    # output size rule of resample_spacing (image_tools.py:363-366)
    assert orz.out_size([100, 100, 40], [0.5, 0.5, 2.0], [1, 1, 1], 16) == [64, 64, 80]
    with pytest.raises(ValueError):
        orz.resample_grid(src, [1, 1, 1], [4, 3, 2], [1, 1, 1], 'CUBIC')


def test_reduced_precision_program_is_the_oracle_when_nothing_is_rounded():
    """oracle/reduced_precision.py with every rounding point switched off (or fp32 'storage') is oracle/net.py."""
    from oracle import reduced_precision as orp
    for arch, cout in (('vnet', 2), ('vbnet', 3)):
        sd = oinit.randomize_affine(oinit.init_state_dict(arch, 1, cout, 0), 2)
        x = torch.randn((1, 1, 16, 16, 32), generator=torch.Generator().manual_seed(4))
        ref = onet.forward(sd, x)
        assert (orp.forward(sd, x, torch.float32) - ref).abs().max() <= 2e-6
        everything = ('in_block', 'down_', 'up_', 'out_block')
        assert (orp.forward(sd, x, torch.float16, exact=everything) - ref).abs().max() <= 2e-6
        y16 = orp.forward(sd, x, torch.float16)
        assert 0 < (y16 - ref).abs().max() <= 1e-2          # fp16 storage: inside BASELINE.json's reduced-precision bar


def test_sliding_window_with_bounding_box_matches_reference():
    """The coarse->fine cascade's call (core/seg_infer.py:292-307,428-444): the box restricts the patch grid; voxels the
    grid never visits have count 0, so the reference leaves NaN probabilities and label 0 there."""
    z = np.load(os.path.join(G, 'cascade.npz'))
    m = json.loads(str(z['meta']))
    sd = oinit.randomize_affine(oinit.init_state_dict(m['arch'], 1, m['cout'], m['wseed']), m['aseed'])
    size = m['size']
    vol = (seeded_input(m['vseed'], (1, 1, size[2], size[1], size[0]), 'smooth')[0, 0].numpy() * m['scale']).astype(np.float32)
    nd = {'type': 0, 'mean': m['norm'][1], 'stddev': m['norm'][2], 'clip': m['norm'][3]}
    with np.errstate(all='ignore'):
        probs, mask, starts, ends = osw.segmentation_volume(sd, vol, [1.0, 1.0, 1.0], nd, 'SIZE', m['psize'], m['pstride'], 16,
                                                            bbox_start_voxel=m['bbox_start'], bbox_end_voxel=m['bbox_end'])
    visited = np.isfinite(z['probs'][0])
    assert 0.3 < visited.mean() < 0.8
    assert np.array_equal(np.isfinite(probs[0]), visited)
    assert np.abs(probs[:, visited] - z['probs'][:, visited]).max() <= 1e-6
    assert np.array_equal(mask, z['mask']) and not mask[~visited].any()
    # the box was rounded up to a multiple of max_stride and shifted back inside the volume (image_tools.py:179-188)
    lo = np.min(np.array(starts), 0).tolist()
    hi = np.max(np.array(ends), 0).tolist()
    zz, yy, xx = np.where(visited)
    assert lo == [int(xx.min()), int(yy.min()), int(zz.min())] and hi == [int(xx.max()) + 1, int(yy.max()) + 1, int(zz.max()) + 1]


CE_CASES = (('ce', {}), ('ce_w', {'weight': True}), ('ce_ign', {'weight': True, 'ignore_index': 1}),
            ('ce_sum', {'reduction': 'sum'}), ('ce_none', {'weight': True, 'ignore_index': 0, 'reduction': 'none'}))


def test_cross_entropy_matches_reference():
    z, zc = np.load(os.path.join(G, 'loss.npz')), np.load(os.path.join(G, 'loss_ce.npz'))
    for c in (2, 5):
        k = 'c%d_' % c
        probs, target = torch.from_numpy(z[k + 'probs']), torch.from_numpy(z[k + 'target'])
        for tag, kw in CE_CASES:
            kw = dict(kw)
            if kw.pop('weight', False):
                kw['weight'] = torch.from_numpy(zc[k + 'weight'])
            p = probs.clone().requires_grad_(True)
            l = oloss.cross_entropy_loss(p, target, **kw)
            (l if l.dim() == 0 else (l * torch.arange(l.numel(), dtype=torch.float32).view_as(l) / l.numel()).sum()).backward()
            assert np.abs(l.detach().numpy() - zc[k + tag]).max() <= 1e-6 * max(1.0, float(np.abs(zc[k + tag]).max())), (k, tag)
            assert np.abs(p.grad.numpy() - zc[k + tag + '_grad']).max() <= 1e-8, (k, tag)
