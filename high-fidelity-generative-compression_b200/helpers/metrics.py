"""PSNR, SSIM and MS-SSIM with the public API of the reference's ``src/helpers/metrics.py``, on the kernels of
``csrc/ssim.cu``.

The names, arguments, defaults, validation order and exception types are the reference's; so are its quirks: trailing
singleton dimensions are squeezed, ``win`` overrides ``win_size``, a spatial dimension smaller than the window is not
smoothed (with the reference's warning), ``ms_ssim`` pools with ``avg_pool2d(kernel 2, padding=s % 2)`` and asserts
``min(H, W) > (win_size - 1) * 16``.

``psnr`` on NumPy arrays (what ``compress.py`` passes) is computed on the host in float64, as the reference does; on CUDA
tensors it returns a per-image float64 tensor computed on the device.  ``ssim`` / ``ms_ssim`` take fp32 CUDA tensors and
return CUDA tensors without synchronising with the host.  What the kernels do not implement raises instead of falling
back: CPU tensors ``RuntimeError``; other dtypes, 5-D inputs, windows longer than 31 taps, more than 8 levels and inputs
that require a gradient ``NotImplementedError`` (these functions are forward-only).
"""
import warnings

import numpy as np
import torch

from .. import ops

MAX_WIN = 31           # csrc/ssim_math.cuh: kSsimMaxWin
MAX_LEVELS = 8         # csrc/ssim_math.cuh: kSsimMaxLevels
_DEFAULT_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def psnr(img1, img2, max_val=255.):
    """Per-image PSNR in dB, ``20 log10(max_val) - 10 log10(mean((img1 - img2)^2))`` over all axes but the first (as
    ``tf.image.psnr``).  NumPy arrays: float64 on the host.  CUDA tensors: a float64 (N,) tensor from the device."""
    if isinstance(img1, torch.Tensor) or isinstance(img2, torch.Tensor):
        if not (isinstance(img1, torch.Tensor) and isinstance(img2, torch.Tensor)):
            raise TypeError("psnr: pass two NumPy arrays or two CUDA tensors")
        if not (img1.is_cuda and img2.is_cuda):
            raise RuntimeError("psnr: tensors must be CUDA tensors (NumPy arrays are computed on the host)")
        if img1.dtype != torch.float32 or img2.dtype != torch.float32:
            raise NotImplementedError(f"psnr: float32 tensors only, got {img1.dtype} and {img2.dtype}")
        if img1.dim() != 4 or img1.shape != img2.shape:
            raise ValueError(f"psnr: two (N, C, H, W) tensors of the same shape expected, got {tuple(img1.shape)} "
                             f"and {tuple(img2.shape)}")
        _no_grad_check(img1, img2, "psnr")
        return ops.psnr(img1, img2, max_val)
    a = np.asarray(img1).astype(np.float64)
    b = np.asarray(img2).astype(np.float64)
    mse = np.mean(np.square(a - b), axis=(1, 2, 3))
    return 20 * np.log10(max_val) - 10 * np.log10(mse)


def _fspecial_gauss_1d(size, sigma):
    """Normalised 1-D Gaussian window of ``size`` taps centred on ``size // 2``, shape (1, 1, size), float32."""
    x = torch.arange(size).to(dtype=torch.float) - size // 2
    g = torch.exp(-(x ** 2) / (2 * sigma ** 2))
    return (g / g.sum()).reshape(1, 1, size)


def _squeeze(X, Y):
    for d in range(X.dim() - 1, 1, -1):
        X, Y = X.squeeze(dim=d), Y.squeeze(dim=d)
    return X, Y


def _no_grad_check(X, Y, what):
    if torch.is_grad_enabled() and (X.requires_grad or Y.requires_grad):
        raise NotImplementedError(f"{what}: forward only -- the CUDA kernels have no backward pass; call it under "
                                  "torch.no_grad() or on detached tensors")


def _require_cuda(X, Y, what):
    if not (X.is_cuda and Y.is_cuda):
        raise RuntimeError(f"{what}: inputs must be CUDA tensors (there is no CPU implementation)")


def _check_supported(X, Y, win_size, what):
    if X.dim() == 5:
        raise NotImplementedError(f"{what}: 5-d (conv3d) inputs are not implemented")
    _require_cuda(X, Y, what)
    if X.dtype != torch.float32:
        raise NotImplementedError(f"{what}: float32 inputs only, got {X.dtype}")
    if win_size > MAX_WIN:
        raise NotImplementedError(f"{what}: window size {win_size} > {MAX_WIN}")
    _no_grad_check(X, Y, what)


_taps_cache = {}


def _device_taps(win, win_size, win_sigma, channels, device):
    """(C, win_size) fp32 taps on `device`.  A CUDA `win` is used as it is; host windows are uploaded once per value and
    device and cached, so a call copies nothing from the host."""
    if win is not None and win.is_cuda:
        if win.shape[0] != channels or win.numel() != channels * win_size:
            raise RuntimeError(f"window of shape {tuple(win.shape)} does not fit {channels} channels")
        return win.detach().reshape(channels, win_size).to(device=device, dtype=torch.float32).contiguous()
    if win is None:
        key = ("gauss", int(win_size), float(win_sigma), channels, device)
    else:
        if win.shape[0] != channels or win.numel() != channels * win_size:
            raise RuntimeError(f"window of shape {tuple(win.shape)} does not fit {channels} channels")
        host = win.detach().reshape(channels, win_size).to(torch.float32).contiguous()
        key = ("taps", host.numpy().tobytes(), channels, win_size, device)
    taps = _taps_cache.get(key)
    if taps is None:
        if win is None:
            host = _fspecial_gauss_1d(win_size, win_sigma).reshape(1, win_size).repeat(channels, 1)
        taps = _taps_cache[key] = host.to(device).contiguous()
    return taps


def _warn_unsmoothed(shape, win_size):
    """The reference's gaussian_filter warning for each spatial dimension smaller than the window."""
    for i, s in enumerate(shape[2:]):
        if s < win_size:
            warnings.warn(f"Skipping Gaussian Smoothing at dimension 2+{i} for input: {shape} and win size: {win_size}")


def _constants(K, data_range):
    K1, K2 = K
    return float((K1 * data_range) ** 2), float((K2 * data_range) ** 2)


def ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, K=(0.01, 0.03),
         nonnegative_ssim=False):
    r"""SSIM of two batches of images (N, C, H, W), fp32 CUDA tensors.

    Args:
        X, Y (torch.Tensor): images
        data_range (float or int): value range of the images (usually 1.0 or 255)
        size_average (bool): average over the batch to a scalar; otherwise one value per image
        win_size (int): Gaussian window length (odd)
        win_sigma (float): Gaussian window sigma
        win (torch.Tensor, optional): (C, 1, 1, win) window taps; overrides win_size / win_sigma
        K (tuple): constants (K1, K2)
        nonnegative_ssim (bool): relu the per-channel SSIM
    Returns:
        torch.Tensor: SSIM (0-d) or (N,)
    """
    if not X.shape == Y.shape:
        raise ValueError("Input images should have the same dimensions.")
    X, Y = _squeeze(X, Y)
    if X.dim() not in (4, 5):
        raise ValueError(f"Input images should be 4-d or 5-d tensors, but got {X.shape}")
    if not X.type() == Y.type():
        raise ValueError("Input images should have the same dtype.")
    if win is not None:
        win_size = win.shape[-1]
    if not (win_size % 2 == 1):
        raise ValueError("Window size should be odd.")
    _check_supported(X, Y, win_size, "ssim")
    _warn_unsmoothed(X.shape, win_size)
    taps = _device_taps(win, win_size, win_sigma, X.shape[1], X.device)
    c1, c2 = _constants(K, data_range)
    return ops.ssim_levels(X, Y, taps, c1, c2, [1.0], bool(nonnegative_ssim), size_average)


def ms_ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, weights=None,
            K=(0.01, 0.03)):
    r"""MS-SSIM of two batches of images (N, C, H, W), fp32 CUDA tensors.

    Args:
        X, Y (torch.Tensor): images
        data_range (float or int): value range of the images (usually 1.0 or 255)
        size_average (bool): average over the batch to a scalar; otherwise one value per image
        win_size (int): Gaussian window length (odd)
        win_sigma (float): Gaussian window sigma
        win (torch.Tensor, optional): (C, 1, 1, win) window taps; overrides win_size / win_sigma
        weights (list, optional): per-level weights; their number is the number of levels
        K (tuple): constants (K1, K2)
    Returns:
        torch.Tensor: MS-SSIM (0-d) or (N,)
    """
    if not X.shape == Y.shape:
        raise ValueError("Input images should have the same dimensions.")
    X, Y = _squeeze(X, Y)
    if not X.type() == Y.type():
        raise ValueError("Input images should have the same dtype.")
    if X.dim() not in (4, 5):
        raise ValueError(f"Input images should be 4-d or 5-d tensors, but got {X.shape}")
    if win is not None:
        win_size = win.shape[-1]
    if not (win_size % 2 == 1):
        raise ValueError("Window size should be odd.")
    smaller_side = min(X.shape[-2:])
    assert smaller_side > (win_size - 1) * (2 ** 4), \
        "Image size should be larger than %d due to the 4 downsamplings in ms-ssim" % ((win_size - 1) * (2 ** 4))
    if weights is None:
        weights = _DEFAULT_WEIGHTS
    weights = [float(w) for w in torch.tensor(weights, dtype=torch.float32).reshape(-1).tolist()]
    if len(weights) > MAX_LEVELS:
        raise NotImplementedError(f"ms_ssim: at most {MAX_LEVELS} levels, got {len(weights)}")
    _check_supported(X, Y, win_size, "ms_ssim")
    shape = X.shape
    for level in range(len(weights)):
        _warn_unsmoothed(shape, win_size)
        shape = torch.Size((shape[0], shape[1], (shape[2] + 1) // 2, (shape[3] + 1) // 2))
    taps = _device_taps(win, win_size, win_sigma, X.shape[1], X.device)
    c1, c2 = _constants(K, data_range)
    return ops.ssim_levels(X, Y, taps, c1, c2, weights, True, size_average)


class SSIM(torch.nn.Module):
    def __init__(self, data_range=255, size_average=True, win_size=11, win_sigma=1.5, channel=3, spatial_dims=2,
                 K=(0.01, 0.03), nonnegative_ssim=False):
        r"""Module form of :func:`ssim`; holds the (channel, 1, 1, win_size) Gaussian window and passes it as ``win``."""
        super().__init__()
        self.win_size = win_size
        self.win = _fspecial_gauss_1d(win_size, win_sigma).repeat([channel, 1] + [1] * spatial_dims)
        self.size_average = size_average
        self.data_range = data_range
        self.K = K
        self.nonnegative_ssim = nonnegative_ssim

    def forward(self, X, Y):
        return ssim(X, Y, data_range=self.data_range, size_average=self.size_average, win=self.win, K=self.K,
                    nonnegative_ssim=self.nonnegative_ssim)


class MS_SSIM(torch.nn.Module):
    def __init__(self, data_range=255, size_average=True, win_size=11, win_sigma=1.5, channel=3, spatial_dims=2,
                 weights=None, K=(0.01, 0.03)):
        r"""Module form of :func:`ms_ssim`; holds the (channel, 1, 1, win_size) Gaussian window and passes it as ``win``."""
        super().__init__()
        self.win_size = win_size
        self.win = _fspecial_gauss_1d(win_size, win_sigma).repeat([channel, 1] + [1] * spatial_dims)
        self.size_average = size_average
        self.data_range = data_range
        self.weights = weights
        self.K = K

    def forward(self, X, Y):
        return ms_ssim(X, Y, data_range=self.data_range, size_average=self.size_average, win=self.win,
                       weights=self.weights, K=self.K)
