"""GPU: the SSIM / MS-SSIM backward kernels (csrc/ssim.cu) behind hific_b200.helpers.metrics_autograd.

  * forward values bit-identical to hific_b200.helpers.metrics;
  * dX and dY against float64 autograd of the oracle: per-image relative L2 <= 5e-5 at the sizes compress.py sees and
    over the case matrix (which input requires a gradient, both reductions, nonnegative_ssim, custom weights / K /
    data_range, the 7-tap window, an input shorter than the window);
  * the golden cases (the reference's float32 CPU gradients): within max(5e-5, 3 x their own distance from float64), and
    exact zeros for the inverted pair;
  * bit-identical gradients on a repeated call and for one image alone vs inside a batch of eight;
  * levels + 1 forward launches, at most 2 * levels + 1 backward launches, none synchronising with the host;
  * end to end: 1 - MS_SSIM on an EVALUATION Model's reconstruction.
"""
import logging
import os
import warnings

import numpy as np
import pytest
import torch

from hific_b200 import ops, synth
from hific_b200.helpers import metrics as M
from hific_b200.helpers import metrics_autograd as MA
from oracle import make_golden_metrics_grad as G
from oracle import metrics_oracle as O

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 5e-5


@pytest.fixture(scope="module")
def src():
    return np.load(G.SRC)


@pytest.fixture(scope="module")
def gold():
    return np.load(G.OUT)


def synth_pair(n, h, w, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (torch.rand((n, 3, h // 16 + 1, w // 16 + 1), device="cuda", generator=g) * 255)
    x = torch.nn.functional.interpolate(x, size=(h, w), mode="bilinear", align_corners=False)
    x = (x + 20 * torch.rand((n, 3, h, w), device="cuda", generator=g)).clamp(0, 255)
    y = (x + 8 * torch.randn((n, 3, h, w), device="cuda", generator=g)).clamp(0, 255)
    return x.contiguous(), y.contiguous()


def rel_l2_per_image(got, want):
    out = []
    for g, w in zip(got.double(), want.double()):
        wn = float(w.norm())
        out.append(float((g - w).norm()) / wn if wn > 0 else (0.0 if not g.any() else float("inf")))
    return out


def kernel_grads(fn, X, Y, need=(True, True), upstream=None):
    Xl, Yl = X.clone().requires_grad_(need[0]), Y.clone().requires_grad_(need[1])
    v = fn(Xl, Yl)
    v.backward(torch.ones_like(v) if upstream is None else upstream)
    return v.detach(), Xl.grad, Yl.grad


def oracle_grads(fn64, X, Y, upstream=None):
    X64, Y64 = X.double().requires_grad_(True), Y.double().requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        v = fn64(X64, Y64)
    v.backward(torch.ones_like(v) if upstream is None else upstream.double())
    return X64.grad, Y64.grad


def assert_close(got, want, bar=TOL):
    assert got is not None and torch.isfinite(got).all()
    err = rel_l2_per_image(got, want)
    assert max(err) <= bar, (err, bar)


def test_forward_is_bit_identical_to_helpers_metrics():
    X, Y = synth_pair(2, 192, 256, 1)
    Xg = X.clone().requires_grad_(True)
    assert torch.equal(MA.ms_ssim(Xg, Y, size_average=False).detach(), M.ms_ssim(X, Y, size_average=False))
    assert torch.equal(MA.MS_SSIM(data_range=255)(Xg, Y).detach(), M.MS_SSIM(data_range=255)(X, Y))
    assert torch.equal(MA.ssim(Xg, Y, nonnegative_ssim=True).detach(), M.ssim(X, Y, nonnegative_ssim=True))
    assert torch.equal(MA.SSIM(win_size=7, size_average=False)(Xg, Y).detach(), M.SSIM(win_size=7, size_average=False)(X, Y))


@pytest.mark.parametrize("n,h,w", [(1, 512, 768), (1, 1365, 2048), (8, 1024, 1024)])
def test_against_float64_autograd_at_compress_sizes(n, h, w):
    X, Y = synth_pair(n, h, w, h + w)
    _, dx, dy = kernel_grads(MA.MS_SSIM(data_range=255), X, Y)
    ox, oy = oracle_grads(lambda a, b: O.ms_ssim(a, b, dtype=torch.float64), X, Y)
    assert_close(dx, ox)
    assert_close(dy, oy)
    del ox, oy
    _, dx, dy = kernel_grads(lambda a, b: MA.ssim(a, b, size_average=False), X, Y)
    ox, oy = oracle_grads(lambda a, b: O.ssim(a, b, size_average=False, dtype=torch.float64), X, Y)
    assert_close(dx, ox)
    assert_close(dy, oy)


def test_golden_cases(src, gold):
    A64 = G.OracleAdapter(torch.float64)
    kernels = {
        "ms": lambda X, Y: MA.ms_ssim(X, Y, data_range=255),
        "sat": lambda X, Y: MA.ms_ssim(X, Y, data_range=255),
        "custom": lambda X, Y: MA.ms_ssim(X, Y, data_range=1, size_average=False, weights=G.W3, K=G.K3).sum(),
        "ssim": lambda X, Y: MA.ssim(X, Y, data_range=255, size_average=False).sum(),
        "ssim_nonneg": lambda X, Y: MA.ssim(X, Y, data_range=255, nonnegative_ssim=True),
        "ssim7": lambda X, Y: MA.ssim(X, Y, data_range=255, win_size=7, win_sigma=1.0),
        "small": lambda X, Y: MA.ssim(X, Y, data_range=255, size_average=False).sum(),
    }
    for case, fn in kernels.items():
        key, scale, loss = G.cases(A64)[case]
        X, Y = (t.cuda() for t in G.inputs(src, key, scale))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            _, dx, dy = kernel_grads(fn, X, Y)
        ox, oy = oracle_grads(loss, X, Y)
        worst = 0.0
        idx = torch.from_numpy(gold[f"{case}.idx"]).long().cuda()
        for name, o in (("dX", ox), ("dY", oy)):
            s = o.reshape(-1)[idx]
            worst = max(worst, float((torch.from_numpy(gold[f"{case}.{name}_sample"]).cuda().double() - s).norm()
                                     / s.norm()))
        bar = max(TOL, 3 * worst)
        assert_close(dx, ox, bar)
        assert_close(dy, oy, bar)
        for name, d in (("dX", dx), ("dY", dy)):
            want = np.sqrt(gold[f"{case}.{name}_sumsq"])
            got = np.sqrt(G.per_image_sumsq(d).cpu().numpy())
            for n, w in zip(got, want):
                assert (n == 0) if w == 0 else abs(n / w - 1) <= bar, (case, name, n, w)
        if case == "ms":
            assert not dx[1].any() and not dy[1].any() and dx[0].abs().sum() > 0     # the inverted pair


CASES = {
    "x_only": (lambda a, b: MA.ms_ssim(a, b), lambda a, b: O.ms_ssim(a, b, dtype=torch.float64), (True, False)),
    "y_only": (lambda a, b: MA.ms_ssim(a, b), lambda a, b: O.ms_ssim(a, b, dtype=torch.float64), (False, True)),
    "per_image": (lambda a, b: MA.ms_ssim(a, b, size_average=False),
                  lambda a, b: O.ms_ssim(a, b, size_average=False, dtype=torch.float64), (True, True)),
    "nonneg": (lambda a, b: MA.ssim(a, b, nonnegative_ssim=True, size_average=False),
               lambda a, b: O.ssim(a, b, size_average=False, nonnegative_ssim=True, dtype=torch.float64), (True, True)),
    "custom": (lambda a, b: MA.ms_ssim(a / 255, b / 255, data_range=1, weights=[0.2, 0.3, 0.5], K=(0.02, 0.4)),
               lambda a, b: O.ms_ssim(a / 255, b / 255, 1, weights=[0.2, 0.3, 0.5], K=(0.02, 0.4), dtype=torch.float64),
               (True, True)),
    "win7": (lambda a, b: MA.MS_SSIM(win_size=7, win_sigma=1.0)(a, b),
             lambda a, b: O.ms_ssim(a, b, taps=O.gauss_taps(7, 1.0), dtype=torch.float64), (True, True)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_case_matrix(case):
    fn, fn64, need = CASES[case]
    X, Y = synth_pair(2, 192, 256, 3)
    up = torch.tensor([0.5, -2.0], device="cuda") if case in ("per_image", "nonneg") else None
    _, dx, dy = kernel_grads(fn, X, Y, need, up)
    ox, oy = oracle_grads(fn64, X, Y, up)
    assert (dx is not None) == need[0] and (dy is not None) == need[1]
    if need[0]:
        assert_close(dx, ox)
    if need[1]:
        assert_close(dy, oy)


def test_unsmoothed_input():
    X, Y = synth_pair(2, 8, 64, 5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _, dx, dy = kernel_grads(lambda a, b: MA.ssim(a, b, size_average=False), X, Y)
    ox, oy = oracle_grads(lambda a, b: O.ssim(a, b, size_average=False, dtype=torch.float64), X, Y)
    assert_close(dx, ox)
    assert_close(dy, oy)


def test_bit_reproducible_and_independent_of_the_batch():
    X, Y = synth_pair(8, 1024, 1024, 11)
    fn = lambda a, b: MA.ms_ssim(a, b, size_average=False)     # noqa: E731
    _, ax, ay = kernel_grads(fn, X, Y)
    _, bx, by = kernel_grads(fn, X, Y)
    assert torch.equal(ax, bx) and torch.equal(ay, by)
    for i in (0, 5):
        _, cx, cy = kernel_grads(fn, X[i:i + 1], Y[i:i + 1])
        assert torch.equal(cx, ax[i:i + 1]) and torch.equal(cy, ay[i:i + 1])


def test_launch_count_and_no_host_synchronisation():
    X, Y = synth_pair(2, 256, 320, 4)
    mod = MA.MS_SSIM(data_range=255)
    for _ in range(2):                                          # warm: the window upload, allocator blocks
        Xl = X.clone().requires_grad_(True)
        mod(Xl, Y).backward()
        Xl = X.clone().requires_grad_(True)
        MA.ssim(Xl, Y).backward()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for fn, levels in ((mod, 5), (lambda a, b: MA.ms_ssim(a, b, weights=[0.2, 0.3, 0.5]), 3), (MA.ssim, 1)):
            Xl, Yl = X.clone().requires_grad_(True), Y.clone().requires_grad_(True)
            l0 = ops.launch_count()
            v = fn(Xl, Yl)
            assert ops.launch_count() - l0 == levels + 1
            l0 = ops.launch_count()
            (1 - v).backward()
            assert ops.launch_count() - l0 <= 2 * levels + 1
    finally:
        torch.cuda.set_sync_debug_mode(0)


def test_end_to_end_through_a_model_reconstruction():
    os.environ.setdefault("HFC_LPIPS_SYNTHETIC", "1")
    from hific_b200.config import ModelModes, mse_lpips_args
    from hific_b200.model import Model
    m = Model(mse_lpips_args(), logging.getLogger("metrics_grad"), model_mode=ModelModes.EVALUATION)
    m.load_state_dict(synth.synth_state_dict(0), strict=False)
    m = m.cuda().eval()
    x = synth.synth_image(1, 192, 256, 7).cuda()
    with torch.no_grad():
        recon = m(x)
        recon = recon[0] if isinstance(recon, tuple) else recon
    recon = recon.detach().clone().requires_grad_(True)
    loss = 1 - MA.MS_SSIM(data_range=255)(recon * 255, x * 255)
    loss.backward()
    r64 = recon.detach().double().requires_grad_(True)
    (1 - O.ms_ssim(r64 * 255, x.double() * 255, dtype=torch.float64)).backward()
    assert_close(recon.grad, r64.grad)
