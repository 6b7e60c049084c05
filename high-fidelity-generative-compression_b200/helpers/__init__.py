"""Mirror of the reference's ``src/helpers`` package: ``metrics`` (PSNR, SSIM, MS-SSIM) on the libhfc kernels."""
