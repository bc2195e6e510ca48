"""Float64 helpers shared by the stage-by-stage tests (test_gpu_train_stages.py, test_gpu_infer_stages.py): elementwise
bounds, float64 copies of the NDHWC channel windows the kernels address, and the GroupNorm scale / shift exactly as the
kernels form it."""
import torch
import torch.nn.functional as F

EPS32 = float(torch.tensor(1e-5, dtype=torch.float32))      # GN_EPS as the kernels receive it


def _close(name, got, ref, mag, rel, frac, absb=0.0, extra=None):
    """|got - ref| <= rel |ref| + frac mag (+ absb + extra) elementwise (NaN fails).  Returns the worst err / bound."""
    got = got.double()
    err = (got - ref).abs()
    tol = rel * ref.abs() + frac * mag
    if absb:
        tol = tol + absb
    if extra is not None:
        tol = tol + extra
    bad = ~(err <= tol)
    if bool(bad.any()):
        excess = torch.where(bad, (err - tol) / (mag + ref.abs() + 1e-300), torch.zeros_like(err))
        excess = torch.nan_to_num(excess, nan=float('inf'))
        i = int(torch.argmax(excess.flatten()))
        raise AssertionError('%s: %d of %d elements out of bound; worst at flat index %d: got %.6g ref %.6g mag %.6g (tol %.3g)'
                             % (name, int(bad.sum()), bad.numel(), i, float(got.flatten()[i]), float(ref.flatten()[i]),
                                float(mag.flatten()[i]), float(tol.flatten()[i])))
    if err.numel() == 0:
        return 0.0
    return float((err / tol.clamp_min(1e-300)).max())


def _rows(v, nvox, b0=0, nb=None):
    """[nb, nvox, C] float64 copy of the channel window (off, C) of an NDHWC buffer with pitch ld, samples [b0, b0 + nb);
    samples are nvox * ld elements apart, as the kernels address them (a buffer may be allocated wider than the view uses)"""
    b = v.buf
    nb = b.shape[0] - b0 if nb is None else nb
    base = v.off + b0 * nvox * v.ld
    assert base + ((nb - 1) * nvox + nvox - 1) * v.ld + v.C <= b.numel(), 'view runs past its buffer'
    return torch.as_strided(b, (nb, nvox, v.C), (nvox * v.ld, v.ld, 1), b.storage_offset() + base).double()


def _window(v, off, C):
    from segmentation3d._b200.plan import _View
    return _View(v.buf, v.off + off, v.ld, C)


def _mean_rstd32(stats, cnt):
    """gn_mean_rstd (csrc/common.cuh): float64 moments, fp32 mean and rstd; [B, 1, 1] float64 holding fp32 values"""
    st = stats.double()
    m = st[:, 0] / cnt
    var = (st[:, 1] / cnt - m * m).clamp_min(0.0)
    rstd = 1.0 / torch.sqrt(var + EPS32)
    return m.float().double().view(-1, 1, 1), rstd.float().double().view(-1, 1, 1)


def _affine32(mean, rstd, gamma, beta):
    """a = fl(rstd * gamma), b = fl(beta - mean * a) with one rounding (FFMA), as the kernels form the ReLU argument"""
    a = (rstd.float() * gamma.float().view(1, 1, -1)).double()
    b = (beta.double().view(1, 1, -1) - mean * a).float().double()
    return a, b


def _taps(k):
    return [(a, b, c) for a in range(k) for b in range(k) for c in range(k)]


def conv_forward(mode, x, w, bias=None):
    """forward convolution as one float64 matmul per tap; x [B, D, H, W, Ci], w in the parameter layout (K3 / K2S2:
    [Co, Ci, k, k, k], T2S2: [Ci, Co, 2, 2, 2]); returns [B, Do, Ho, Wo, Co]"""
    from segmentation3d._b200 import lib
    B, D, H, W, Ci = x.shape
    if mode == lib.CONV_T2S2:
        Co = w.shape[1]
        out = x.new_zeros((B, 2 * D, 2 * H, 2 * W, Co))
        x2 = x.reshape(-1, Ci)
        for (a, b, c) in _taps(2):
            out[:, a::2, b::2, c::2] = (x2 @ w[:, :, a, b, c]).view(B, D, H, W, Co)
    elif mode == lib.CONV_K2S2:
        Co = w.shape[0]
        out = x.new_zeros((B, D // 2, H // 2, W // 2, Co))
        for (a, b, c) in _taps(2):
            out += (x[:, a::2, b::2, c::2].reshape(-1, Ci) @ w[:, :, a, b, c].t()).view(out.shape)
    else:
        Co = w.shape[0]
        xp = F.pad(x, (0, 0, 1, 1, 1, 1, 1, 1))
        out = x.new_zeros((B, D, H, W, Co))
        for (a, b, c) in _taps(3):
            out += (xp[:, a:a + D, b:b + H, c:c + W].reshape(-1, Ci) @ w[:, :, a, b, c].t()).view(out.shape)
        del xp
    if bias is not None:
        out += bias.double().view(1, 1, 1, 1, -1)
    return out
