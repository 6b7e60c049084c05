"""Restatement of the reference's image-quality metrics (src/helpers/metrics.py) in torch, for any dtype and device --
TEST INFRASTRUCTURE.

float32 on the CPU, with the thread count of tests/golden/metrics.npz (THREADS), reproduces the reference's stored outputs
bit for bit: it issues the same conv2d / avg_pool2d calls and the same element-wise expressions in the same order.
float64 is the comparator for sizes too large to store (the window taps stay the reference's float32 values, widened).
On a GPU the float32 form is the reference formulation the benchmark times (tools/metrics_bench.py).
"""
import numpy as np
import torch
import torch.nn.functional as F

THREADS = 8
DEFAULT_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def gauss_taps(win_size=11, win_sigma=1.5):
    """The reference's float32 Gaussian window, (win_size,)."""
    d = torch.arange(win_size, dtype=torch.float32) - win_size // 2
    e = torch.exp(-(d ** 2) / (2 * win_sigma ** 2))
    return e / e.sum()


def _smooth(x, taps):
    """Separable valid-mode filter: along H, then along W; a dimension shorter than the window is left as it is."""
    c, k = x.shape[1], taps.numel()
    w = taps.reshape(1, 1, 1, k).expand(c, 1, 1, k).to(x.device, x.dtype)
    if x.shape[2] >= k:
        x = F.conv2d(x, w.transpose(2, 3), groups=c)
    if x.shape[3] >= k:
        x = F.conv2d(x, w, groups=c)
    return x


def level_stats(X, Y, taps, data_range=255, K=(0.01, 0.03)):
    """(ssim, cs) per (image, channel) of one level."""
    C1, C2 = (K[0] * data_range) ** 2, (K[1] * data_range) ** 2
    m1, m2 = _smooth(X, taps), _smooth(Y, taps)
    m1s, m2s, m12 = m1.pow(2), m2.pow(2), m1 * m2
    v1 = _smooth(X * X, taps) - m1s
    v2 = _smooth(Y * Y, taps) - m2s
    v12 = _smooth(X * Y, taps) - m12
    cs = (2 * v12 + C2) / (v1 + v2 + C2)
    s = ((2 * m12 + C1) / (m1s + m2s + C1)) * cs
    return s.flatten(2).mean(-1), cs.flatten(2).mean(-1)


def pool(x):
    return F.avg_pool2d(x, kernel_size=2, padding=[s % 2 for s in x.shape[2:]])


def ms_ssim_levels(X, Y, taps, data_range=255, K=(0.01, 0.03), levels=5):
    """[(ssim, cs)] per level, each (N, C)."""
    out = []
    for level in range(levels):
        out.append(level_stats(X, Y, taps, data_range, K))
        if level < levels - 1:
            X, Y = pool(X), pool(Y)
    return out


def ms_ssim(X, Y, data_range=255, size_average=True, taps=None, weights=None, K=(0.01, 0.03), dtype=torch.float32):
    taps = gauss_taps() if taps is None else taps
    w = torch.tensor(DEFAULT_WEIGHTS if weights is None else weights, dtype=torch.float32).to(X.device, dtype)
    X, Y = X.to(dtype), Y.to(dtype)
    stats = ms_ssim_levels(X, Y, taps, data_range, K, w.numel())
    vals = [torch.relu(cs) for _, cs in stats[:-1]] + [torch.relu(stats[-1][0])]
    v = torch.prod(torch.stack(vals) ** w.view(-1, 1, 1), dim=0)
    return v.mean() if size_average else v.mean(1)


def ssim(X, Y, data_range=255, size_average=True, taps=None, K=(0.01, 0.03), nonnegative_ssim=False,
         dtype=torch.float32):
    taps = gauss_taps() if taps is None else taps
    s, _ = level_stats(X.to(dtype), Y.to(dtype), taps, data_range, K)
    if nonnegative_ssim:
        s = torch.relu(s)
    return s.mean() if size_average else s.mean(1)


def psnr(a, b, max_val=255.0):
    """float64 per-image PSNR of two arrays / tensors (N, ...)."""
    a = np.asarray(a.cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    b = np.asarray(b.cpu() if isinstance(b, torch.Tensor) else b, dtype=np.float64)
    mse = np.square(a - b).reshape(a.shape[0], -1).mean(axis=1)
    return 20 * np.log10(max_val) - 10 * np.log10(mse)
