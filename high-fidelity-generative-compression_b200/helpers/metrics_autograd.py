"""Differentiable SSIM and MS-SSIM with the public API of the reference's ``src/helpers/metrics.py``, on the kernels of
``csrc/ssim.cu``.

Same names, signatures, defaults, validation order, exception types and warnings as :mod:`hific_b200.helpers.metrics`
(the two modules share that code), but ``ssim`` / ``ms_ssim`` / ``SSIM`` / ``MS_SSIM`` have a gradient with respect to
``X`` and ``Y``, so a codec can be trained or fine-tuned on ``1 - ms_ssim(x_hat, x)``.  The forward values are
bit-identical to :mod:`hific_b200.helpers.metrics`; the backward runs at most ``2 * levels + 1`` kernels, does not
synchronise with the host and is bit-reproducible.  Each call that needs a gradient keeps its own workspace and pooled
pyramid until its backward.  Not differentiable: the window (a ``win`` that requires a gradient raises
``NotImplementedError``), a second backward through the gradient (``once_differentiable``) and ``psnr``, which is
re-exported unchanged (the reference's is NumPy).

Reference code that trains through MS-SSIM picks this module up with::

    sys.modules["src.helpers.metrics"] = hific_b200.helpers.metrics_autograd
"""
import torch

from .. import ops
from . import metrics as _m
from .metrics import _fspecial_gauss_1d, psnr  # noqa: F401  (re-exported unchanged)

MAX_WIN = _m.MAX_WIN
MAX_LEVELS = _m.MAX_LEVELS


def ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, K=(0.01, 0.03),
         nonnegative_ssim=False):
    r"""SSIM of two batches of images (N, C, H, W), fp32 CUDA tensors, differentiable with respect to X and Y.

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
    X, Y, taps, c1, c2 = _m._ssim_inputs(X, Y, data_range, win_size, win_sigma, win, K, forward_only=False)
    return ops.ssim_levels_grad(X, Y, taps, c1, c2, [1.0], bool(nonnegative_ssim), size_average)


def ms_ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, weights=None,
            K=(0.01, 0.03)):
    r"""MS-SSIM of two batches of images (N, C, H, W), fp32 CUDA tensors, differentiable with respect to X and Y.

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
    X, Y, taps, c1, c2, weights = _m._ms_ssim_inputs(X, Y, data_range, win_size, win_sigma, win, weights, K,
                                                     forward_only=False)
    return ops.ssim_levels_grad(X, Y, taps, c1, c2, weights, True, size_average)


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
