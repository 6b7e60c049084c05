"""GPU: the PSNR / SSIM / MS-SSIM kernels (csrc/ssim.cu) behind hific_b200.helpers.metrics.

  * every case of tests/golden/metrics.npz (the reference's float32 CPU outputs): SSIM / MS-SSIM within 2e-6, PSNR
    within 1e-6 dB;
  * the float64 oracle at the sizes compress.py sees, same tolerances;
  * bit-identical results on a repeated call and for one image alone vs inside a batch of eight;
  * levels + 1 launches (ssim: 2), none of them synchronising with the host;
  * end to end: Model.compress -> decompress, then MS_SSIM and psnr on the CUDA reconstruction.
"""
import logging
import os
import warnings

import numpy as np
import pytest
import torch

from hific_b200 import ops, synth
from hific_b200.helpers import metrics as M
from oracle import metrics_oracle as O

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

HERE = os.path.dirname(os.path.abspath(__file__))
TOL, TOL_DB = 2e-6, 1e-6
W3, K3 = [0.2, 0.3, 0.5], (0.01, 0.4)


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(HERE, "golden", "metrics.npz"))


def pair(gold, key, scale=1.0):
    return tuple((torch.from_numpy(gold[f"{key}.{s}"]).float() * scale).cuda() for s in ("x", "y"))


def close(got, want, tol=TOL):
    got = got.detach().cpu().numpy().astype(np.float64)
    want = np.asarray(want.cpu() if isinstance(want, torch.Tensor) else want, dtype=np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    err = float(np.max(np.abs(got - want)))
    assert err <= tol, err


def test_golden_cases(gold):
    for key in ("ms", "sat"):
        X, Y = pair(gold, key)
        close(M.MS_SSIM(data_range=255)(X, Y), gold[f"{key}.ms_ssim"])
        close(M.ms_ssim(X, Y, data_range=255, size_average=False), gold[f"{key}.ms_ssim_per_image"])
        close(M.psnr(X, Y, 255.), gold[f"{key}.psnr"], TOL_DB)
        assert M.psnr(X, Y).dtype == torch.float64
    X, Y = pair(gold, "ms", 1 / 255.0)
    close(M.ms_ssim(X, Y, data_range=1, size_average=False, weights=W3, K=K3), gold["custom.ms_ssim_per_image"])
    close(M.psnr(X, Y, 1.), gold["custom.psnr"], TOL_DB)
    X, Y = pair(gold, "ms")
    close(M.ssim(X, Y, nonnegative_ssim=True), gold["ms.ssim_nonneg"])
    close(M.ssim(X, Y, nonnegative_ssim=True, size_average=False), gold["ms.ssim_nonneg_per_image"])
    for key in ("ms", "sat"):
        X, Y = pair(gold, key)
        close(M.ssim(X, Y, size_average=False), gold[f"{key}.ssim_per_image"])
        close(M.SSIM(win_size=7, win_sigma=1.0, size_average=False)(X, Y), gold[f"{key}.ssim7_per_image"])
    X, Y = pair(gold, "small")
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        close(M.ssim(X, Y, size_average=False), gold["small.ssim_per_image"])
    assert [str(w.message) for w in caught] == [str(gold["small.warning"])]
    close(M.psnr(X, Y), gold["small.psnr"], TOL_DB)


def test_pooled_planes_match_avg_pool2d():
    """The level kernel's pooled outputs (the next level's inputs) against F.avg_pool2d, odd sizes."""
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.rand((2, 3, 177, 243), device="cuda", generator=g) * 255
    y = torch.rand((2, 3, 177, 243), device="cuda", generator=g) * 255
    taps = O.gauss_taps().reshape(1, 11).repeat(3, 1).cuda()
    ws, ws_bytes = ops._metrics_ws("ssim", int(ops.lib.hfc_ssim_ws_bytes(2, 3, 177, 243, 11, 2)), x.device)
    px, py = torch.empty((2, 3, 89, 122), device="cuda"), torch.empty((2, 3, 89, 122), device="cuda")
    ops.check(ops.lib.hfc_ssim_level(ops._ptr(x), ops._ptr(y), 2, 3, 177, 243, 0, ops._ptr(taps), 11, 6.5025, 58.5225,
                                     ops._ptr(px), ops._ptr(py), ops._ptr(ws), ws_bytes, ops._stream()), "ssim_level")
    for got, src in ((px, x), (py, y)):
        want = O.pool(src)
        assert torch.allclose(got, want, rtol=2 ** -23, atol=0)


def synth_pair(n, h, w, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (torch.rand((n, 3, h // 16 + 1, w // 16 + 1), device="cuda", generator=g) * 255)
    x = torch.nn.functional.interpolate(x, size=(h, w), mode="bilinear", align_corners=False)
    x = (x + 20 * torch.rand((n, 3, h, w), device="cuda", generator=g)).clamp(0, 255)
    y = (x + 8 * torch.randn((n, 3, h, w), device="cuda", generator=g)).clamp(0, 255)
    return x.contiguous(), y.contiguous()


@pytest.mark.parametrize("n,h,w", [(1, 512, 768), (1, 1365, 2048), (8, 1024, 1024)])
def test_against_the_float64_oracle_at_compress_sizes(n, h, w):
    X, Y = synth_pair(n, h, w, h + w)
    close(M.ms_ssim(X, Y, size_average=False), O.ms_ssim(X, Y, size_average=False, dtype=torch.float64))
    close(M.MS_SSIM(data_range=255)(X, Y), O.ms_ssim(X, Y, dtype=torch.float64))
    close(M.ssim(X, Y, size_average=False), O.ssim(X, Y, size_average=False, dtype=torch.float64))
    close(M.psnr(X, Y), O.psnr(X, Y), TOL_DB)


def test_bit_reproducible_and_independent_of_the_batch():
    X, Y = synth_pair(8, 1024, 1024, 11)
    a = M.ms_ssim(X, Y, size_average=False)
    b = M.ms_ssim(X, Y, size_average=False)
    assert torch.equal(a, b)
    assert torch.equal(M.psnr(X, Y), M.psnr(X, Y))
    assert torch.equal(M.ssim(X, Y, size_average=False), M.ssim(X, Y, size_average=False))
    for i in (0, 5):
        assert torch.equal(M.ms_ssim(X[i:i + 1], Y[i:i + 1], size_average=False), a[i:i + 1])
        assert torch.equal(M.psnr(X[i:i + 1], Y[i:i + 1]), M.psnr(X, Y)[i:i + 1])


def test_launch_count_and_no_host_synchronisation():
    X, Y = synth_pair(2, 256, 320, 4)
    mod, mod7 = M.MS_SSIM(data_range=255), M.SSIM(win_size=7)
    mod(X, Y), mod7(X, Y), M.ssim(X, Y), M.psnr(X, Y)    # warm: the one upload of each window, the workspaces
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        l0 = ops.launch_count()
        mod(X, Y)
        assert ops.launch_count() - l0 == 5 + 1
        l0 = ops.launch_count()
        M.ms_ssim(X, Y, weights=W3)
        assert ops.launch_count() - l0 == 3 + 1
        l0 = ops.launch_count()
        M.ssim(X, Y, size_average=False)
        assert ops.launch_count() - l0 == 2
        mod7(X, Y)
        M.psnr(X, Y)
    finally:
        torch.cuda.set_sync_debug_mode(0)


def test_end_to_end_after_compress_decompress():
    os.environ.setdefault("HFC_LPIPS_SYNTHETIC", "1")
    from hific_b200.config import ModelModes, mse_lpips_args
    from hific_b200.model import Model
    gold = np.load(os.path.join(HERE, "golden", "entropy_coding.npz"))
    m = Model(mse_lpips_args(), logging.getLogger("metrics"), model_mode=ModelModes.EVALUATION)
    m.load_state_dict(synth.synth_state_dict(0), strict=False)
    m.Hyperprior.hyperprior_entropy_model._register_tables(gold["hyper.CDF"], gold["hyper.CDF_offset"],
                                                           gold["hyper.CDF_length"])
    m = m.cuda().eval()
    x = synth.synth_image(1, 192, 256, 7).cuda()
    with torch.no_grad():
        recon = m.decompress(m.compress(x, silent=True))
    a, b = recon * 255.0, x * 255.0
    close(M.MS_SSIM(data_range=255)(a, b), O.ms_ssim(a, b, dtype=torch.float64))
    close(M.psnr(a.contiguous(), b.contiguous(), 255.), O.psnr(a, b, 255.), TOL_DB)
