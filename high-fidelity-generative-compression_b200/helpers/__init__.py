"""Mirror of the reference's ``src/helpers`` package: ``metrics`` (PSNR, SSIM, MS-SSIM) on the libhfc kernels,
forward-only; ``metrics_autograd``, the same API with gradients of SSIM and MS-SSIM."""
