"""CPU: gradients of SSIM / MS-SSIM (src/helpers/metrics.py) against tests/golden/metrics_grad.npz
(oracle/make_golden_metrics_grad.py).

  * the oracle restatement's autograd (oracle/metrics_oracle.py) reproduces the reference's stored gradients bit for bit;
  * the backward's element code (csrc/ssim_math.cuh, compiled with g++ through tests/ssim_grad_host.cpp) gives whole-image
    dX and dY for every golden case within the GPU tests' tolerance of float64 autograd of the oracle, exact zeros for
    the inverted pair, and writes every input pixel of every level from exactly one tile;
  * the host glue of hific_b200.helpers.metrics_autograd and ops.SsimLevelsFn, with a CPU stand-in for the launches:
    validation identical to helpers.metrics, gradients only where asked, no double backward, no window gradient, and
    one workspace per call.
The kernels themselves are checked by tests/test_gpu_metrics_grad.py on a GPU.
"""
import ctypes
import os
import subprocess
import warnings

import numpy as np
import pytest
import torch

from oracle import make_golden_metrics_grad as G
from oracle import metrics_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 5e-5
# case -> (data_range, K, weights, relu_last, size_average, win, sigma); the input key and loss are G.cases()
PARAMS = {
    "ms": (255, (0.01, 0.03), O.DEFAULT_WEIGHTS, 1, 1, 11, 1.5),
    "sat": (255, (0.01, 0.03), O.DEFAULT_WEIGHTS, 1, 1, 11, 1.5),
    "custom": (1, G.K3, G.W3, 1, 0, 11, 1.5),
    "ssim": (255, (0.01, 0.03), [1.0], 0, 0, 11, 1.5),
    "ssim_nonneg": (255, (0.01, 0.03), [1.0], 1, 1, 11, 1.5),
    "ssim7": (255, (0.01, 0.03), [1.0], 0, 1, 7, 1.0),
    "small": (255, (0.01, 0.03), [1.0], 0, 0, 11, 1.5),
}


@pytest.fixture(scope="module")
def src():
    return np.load(G.SRC)


@pytest.fixture(scope="module")
def gold():
    return np.load(G.OUT)


@pytest.fixture
def oracle_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(O.THREADS)
    yield
    torch.set_num_threads(n)


def test_golden_file_is_small_and_complete(gold):
    assert os.path.getsize(G.OUT) <= 256 * 1024
    for case in PARAMS:
        for k in ("idx", "dX_sample", "dY_sample", "dX_sumsq", "dY_sumsq"):
            assert f"{case}.{k}" in gold.files, (case, k)
        assert gold[f"{case}.idx"].size == (G.SAMPLE_LARGE if case in G.LARGE else G.SAMPLE)


def test_oracle_autograd_reproduces_the_reference_bit_for_bit(src, gold, oracle_threads):
    A = G.OracleAdapter()
    for case in PARAMS:
        dX, dY = G.grads(A, src, case)
        idx = torch.from_numpy(gold[f"{case}.idx"]).long()
        for name, g in (("dX", dX), ("dY", dY)):
            assert np.array_equal(g.reshape(-1)[idx].numpy(), gold[f"{case}.{name}_sample"]), (case, name)
            assert np.array_equal(G.per_image_sumsq(g).numpy(), gold[f"{case}.{name}_sumsq"]), (case, name)
    # the inverted pair of `ms`: exactly zero
    assert gold["ms.dX_sumsq"][1] == 0 and gold["ms.dY_sumsq"][1] == 0 and gold["ms.dX_sumsq"][0] > 0


def rel_l2_per_image(got, want):
    """Per-image relative L2 distance; an image whose wanted gradient is exactly 0 must be exactly 0."""
    out = []
    for g, w in zip(got.double(), want.double()):
        wn = float(w.norm())
        out.append(float((g - w).norm()) / wn if wn > 0 else (0.0 if not g.any() else float("inf")))
    return out


def reference_bar(gold, case, d64):
    """max(TOL, 3 x the stored float32 reference gradients' distance from float64, over the stored sample)."""
    worst = 0.0
    idx = torch.from_numpy(gold[f"{case}.idx"]).long()
    for name, w64 in zip(("dX", "dY"), d64):
        ws = w64.reshape(-1)[idx]
        worst = max(worst, float((torch.from_numpy(gold[f"{case}.{name}_sample"]).double() - ws).norm() / ws.norm()))
    return max(TOL, 3 * worst)


def assert_norms_match_reference(gold, case, dx, dy, bar):
    """Per-image L2 norms of the whole gradients against the reference's stored sums of squares (exact 0 stays 0)."""
    for name, got in (("dX", dx), ("dY", dy)):
        want = np.sqrt(gold[f"{case}.{name}_sumsq"])
        norms = np.sqrt(G.per_image_sumsq(got.cpu()).numpy())
        for n, w in zip(norms, want):
            assert (n == 0) if w == 0 else abs(n / w - 1) <= bar, (case, name, n, w)


# ---------------------------------------------------------------------------------------------------------------------
# the backward's element code on the host
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("ssim_grad") / "ssim_grad_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-x", "c++",
                    os.path.join(HERE, "ssim_grad_host.cpp"), "-o", so], check=True)
    return ctypes.CDLL(so)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def level_sizes(h, w, levels):
    out = []
    for _ in range(levels):
        out.append((h, w))
        h, w = (h + 1) // 2, (w + 1) // 2
    return out


def host_grad(host, X, Y, taps, data_range, K, weights, relu_last, size_average, grad_out):
    """Whole backward on the host; returns (dX, dY) and checks that every input pixel of every level has one owner."""
    n, c, h, w = X.shape
    win = taps.numel()
    levels = len(weights)
    x, y = X.float().contiguous(), Y.float().contiguous()
    tap_table = taps.reshape(1, win).repeat(c, 1).float().contiguous()
    sizes = level_sizes(h, w, levels)
    cover = torch.zeros(sum(n * c * a * b for a, b in sizes), dtype=torch.int32)
    dx, dy = torch.empty_like(x), torch.empty_like(y)
    wts = (ctypes.c_float * levels)(*weights)
    g = grad_out.float().contiguous()
    host.ssim_grad_host(_p(x), _p(y), n * c, c, h, w, levels, _p(tap_table), win,
                        ctypes.c_float((K[0] * data_range) ** 2), ctypes.c_float((K[1] * data_range) ** 2), wts,
                        relu_last, size_average, _p(g), _p(dx), _p(dy), _p(cover))
    assert bool((cover == 1).all()), "input pixels not owned by exactly one level-backward tile"
    return dx, dy


def test_host_backward_on_golden_cases(host, src, gold):
    for case, (dr, K, weights, relu_last, size_average, win, sigma) in PARAMS.items():
        key, scale, _ = G.cases(None)[case]
        X, Y = G.inputs(src, key, scale)
        d64 = G.grads(G.OracleAdapter(torch.float64), src, case, torch.float64)
        g = torch.ones(1 if size_average else X.shape[0])
        dx, dy = host_grad(host, X, Y, O.gauss_taps(win, sigma), dr, K, list(weights), relu_last, size_average, g)
        bar = reference_bar(gold, case, d64)
        for got, want in ((dx, d64[0]), (dy, d64[1])):
            assert torch.isfinite(got).all(), case
            err = rel_l2_per_image(got, want)
            assert max(err) <= bar, (case, err, bar)
        assert_norms_match_reference(gold, case, dx, dy, bar)
    # the inverted pair of `ms`: cs < 0 at every level, so its MS-SSIM gradient is exactly 0
    X, Y = G.inputs(src, "ms", 1.0)
    dx, dy = host_grad(host, X, Y, O.gauss_taps(), 255, (0.01, 0.03), list(O.DEFAULT_WEIGHTS), 1, 0, torch.ones(2))
    assert not dx[1].any() and not dy[1].any() and dx[0].abs().sum() > 0


def test_host_backward_per_image_upstream_and_odd_sizes(host):
    """Odd sizes at several levels, small windows and a window longer than the coarse levels (not smoothed there), with
    a per-image upstream gradient; every level's input pixels are written exactly once (checked in host_grad)."""
    gen = torch.Generator().manual_seed(7)
    for h, w, win, levels in ((177, 243, 11, 3), (97, 161, 3, 4), (35, 31, 31, 3), (1, 1, 1, 2), (70, 130, 5, 5)):
        X = torch.rand((2, 2, h, w), generator=gen) * 255
        Y = (X + 20 * torch.randn(X.shape, generator=gen)).clamp(0, 255)
        weights = [0.5 + 0.25 * l for l in range(levels)]
        taps = O.gauss_taps(win, 1.5)
        g = torch.tensor([0.75, -1.5])
        dx, dy = host_grad(host, X, Y, taps, 255, (0.01, 0.03), weights, 1, 0, g)
        X64, Y64 = X.double().requires_grad_(True), Y.double().requires_grad_(True)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            stats = O.ms_ssim_levels(X64, Y64, taps, 255, (0.01, 0.03), levels)
        vals = [torch.relu(cs) for _, cs in stats[:-1]] + [torch.relu(stats[-1][0])]
        wt = torch.tensor(weights, dtype=torch.float32).double().view(-1, 1, 1)
        v = torch.prod(torch.stack(vals) ** wt, dim=0).mean(1)
        (v * g.double()).sum().backward()
        for got, want in ((dx, X64.grad), (dy, Y64.grad)):
            err = rel_l2_per_image(got, want)
            assert max(err) <= TOL, ((h, w, win, levels), err)


# ---------------------------------------------------------------------------------------------------------------------
# host glue of hific_b200.helpers.metrics_autograd and ops.SsimLevelsFn, with a CPU stand-in for the launches
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_value(x, y, taps, c1, c2, weights, relu_last, size_average):
    vals = None
    t = taps[0]
    for level, w in enumerate(weights):
        m1, m2 = O._smooth(x, t), O._smooth(y, t)
        m1s, m2s, m12 = m1.pow(2), m2.pow(2), m1 * m2
        v1, v2, v12 = O._smooth(x * x, t) - m1s, O._smooth(y * y, t) - m2s, O._smooth(x * y, t) - m12
        cs_map = (2 * v12 + c2) / (v1 + v2 + c2)
        s = (((2 * m12 + c1) / (m1s + m2s + c1)) * cs_map).flatten(2).mean(-1)
        cs = cs_map.flatten(2).mean(-1)
        last = level == len(weights) - 1
        v = (torch.relu(s) if relu_last else s) if last else torch.relu(cs)
        f = v ** w
        vals = f if vals is None else vals * f
        if not last:
            x, y = O.pool(x), O.pool(y)
    return vals.mean() if size_average else vals.mean(1)


class CpuLaunches:
    """Stand-in for ops' forward and backward launch sequences.  The forward leaves a fingerprint of its inputs in the
    workspace it is given, and the backward checks that the workspace it reads still holds it."""

    def __init__(self):
        self.backward_calls = []

    def forward(self, x, y, taps, c1, c2, weights, relu_last, size_average, ws, ws_bytes):
        with torch.no_grad():
            out = _oracle_value(x, y, taps, c1, c2, weights, relu_last, size_average)
            ws[0], ws[1] = float(x.double().sum()), float(y.double().sum())
            pyramid = [(x, y)]
            for _ in range(len(weights) - 1):
                pyramid.append((O.pool(pyramid[-1][0]), O.pool(pyramid[-1][1])))
        return out, pyramid

    def backward(self, pyramid, taps, c1, c2, weights, relu_last, size_average, ws, ws_bytes, grad_out, need_x,
                 need_y):
        x, y = pyramid[0]
        assert float(ws[0]) == float(x.double().sum()) and float(ws[1]) == float(y.double().sum()), \
            "workspace overwritten between forward and backward"
        self.backward_calls.append((need_x, need_y))
        xl, yl = x.detach().clone().requires_grad_(need_x), y.detach().clone().requires_grad_(need_y)
        with torch.enable_grad():
            v = _oracle_value(xl, yl, taps, c1, c2, weights, relu_last, size_average)
            grads = torch.autograd.grad(v, [t for t in (xl, yl) if t.requires_grad], grad_out)
        grads = list(grads)
        return (grads.pop(0) if need_x else None), (grads.pop(0) if need_y else None)


@pytest.fixture
def MA(monkeypatch):
    from hific_b200 import ops
    from hific_b200.helpers import metrics, metrics_autograd
    fake = CpuLaunches()
    monkeypatch.setattr(ops, "_ssim_forward_launches", fake.forward)
    monkeypatch.setattr(ops, "_ssim_backward_launches", fake.backward)
    monkeypatch.setattr(ops, "_ssim_check_args", lambda x, y, taps: None)
    monkeypatch.setattr(metrics, "_require_cuda", lambda X, Y, what: None)
    metrics_autograd.fake = fake
    return metrics_autograd


def test_public_names():
    from hific_b200.helpers import metrics, metrics_autograd
    for name in ("psnr", "ssim", "ms_ssim", "SSIM", "MS_SSIM", "_fspecial_gauss_1d"):
        assert hasattr(metrics_autograd, name)
    assert metrics_autograd.psnr is metrics.psnr and metrics_autograd._fspecial_gauss_1d is metrics._fspecial_gauss_1d
    assert metrics_autograd.SSIM(channel=3).win.shape == (3, 1, 1, 11)
    assert metrics_autograd.MS_SSIM(channel=4).win.shape == (4, 1, 1, 11)


def _outcome(fn, *args, **kw):
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        try:
            fn(*args, **kw)
            err = None
        except Exception as e:        # noqa: BLE001 -- the exception itself is what is compared
            err = (type(e), str(e))
    return err, [str(w.message) for w in caught]


def test_validation_is_identical_to_helpers_metrics(MA):
    from hific_b200.helpers import metrics
    X = torch.rand((1, 3, 176, 176))
    bad = torch.rand((3, 176, 176))
    small = torch.rand((1, 3, 160, 200))
    calls = [
        ("ssim", (X, X[:, :2]), {}), ("ms_ssim", (X, X[:, :2]), {}),
        ("ssim", (bad, bad), {}), ("ms_ssim", (bad, bad), {}),
        ("ssim", (X, X.double()), {}), ("ms_ssim", (X, X.double()), {}),
        ("ssim", (bad, bad.double()), {}), ("ms_ssim", (bad, bad.double()), {}),
        ("ssim", (X, X), {"win_size": 10}), ("ms_ssim", (X, X), {"win": torch.ones(3, 1, 1, 4)}),
        ("ms_ssim", (small, small), {}), ("ms_ssim", (torch.rand((1, 3, 96, 200)),) * 2, {"win_size": 7}),
        ("ssim", (X.double(), X.double()), {}), ("ms_ssim", (X.double(), X.double()), {}),
        ("ssim", (torch.rand((1, 3, 4, 176, 176)),) * 2, {}), ("ms_ssim", (torch.rand((1, 3, 4, 176, 176)),) * 2, {}),
        ("ssim", (torch.rand((1, 3, 600, 600)),) * 2, {"win_size": 33}),
        ("ms_ssim", (X, X), {"weights": [0.1] * 9}),
        ("ssim", (torch.rand((2, 3, 8, 64)),) * 2, {}),                          # the unsmoothed-dimension warning
        ("ms_ssim", (torch.rand((1, 3, 200, 176)),) * 2, {"weights": [0.125] * 8}),   # warnings at coarse levels
    ]
    for name, args, kw in calls:
        want = _outcome(getattr(metrics, name), *args, **kw)
        got = _outcome(getattr(MA, name), *args, **kw)
        assert got == want, (name, kw, got, want)
    assert _outcome(MA.ssim, *calls[-2][1])[1] and _outcome(MA.ms_ssim, *calls[-1][1], **calls[-1][2])[1]
    # what differs: a gradient is allowed here, forward-only there
    Xg = X.clone().requires_grad_(True)
    assert _outcome(metrics.ssim, Xg, X)[0][0] is NotImplementedError
    assert _outcome(MA.ssim, Xg, X)[0] is None


def test_gradients_only_where_asked(MA):
    gen = torch.Generator().manual_seed(1)
    X = torch.rand((2, 3, 176, 180), generator=gen) * 255
    Y = (X + 5 * torch.randn(X.shape, generator=gen)).clamp(0, 255)
    for need_x, need_y in ((True, False), (False, True), (True, True)):
        Xl, Yl = X.clone().requires_grad_(need_x), Y.clone().requires_grad_(need_y)
        MA.fake.backward_calls.clear()
        (1 - MA.ms_ssim(Xl, Yl, data_range=255)).backward()
        assert MA.fake.backward_calls == [(need_x, need_y)]
        assert (Xl.grad is not None) == need_x and (Yl.grad is not None) == need_y
    # no gradient asked for: the forward-only path, no backward state
    with torch.no_grad():
        v = MA.ssim(X.clone().requires_grad_(True), Y)
    assert not v.requires_grad
    assert not MA.ssim(X, Y).requires_grad


def test_gradient_matches_autograd_of_the_oracle(MA):
    gen = torch.Generator().manual_seed(2)
    X = torch.rand((2, 3, 176, 180), generator=gen) * 255
    Y = (X + 5 * torch.randn(X.shape, generator=gen)).clamp(0, 255)
    Xl = X.clone().requires_grad_(True)
    MA.SSIM(data_range=255, size_average=False, nonnegative_ssim=True)(Xl, Y).sum().backward()
    Xr = X.clone().requires_grad_(True)
    O.ssim(Xr, Y, size_average=False, nonnegative_ssim=True).sum().backward()
    assert torch.allclose(Xl.grad, Xr.grad, rtol=1e-5, atol=1e-9)


def test_double_backward_raises(MA):
    X = (torch.rand((1, 3, 176, 176)) * 255).requires_grad_(True)
    Y = torch.rand((1, 3, 176, 176)) * 255
    v = MA.ms_ssim(X, Y)
    (g,) = torch.autograd.grad(v, X, grad_outputs=torch.ones_like(v, requires_grad=True), create_graph=True)
    with pytest.raises(RuntimeError, match="differentiate twice"):
        g.sum().backward()


def test_window_that_requires_grad_raises(MA):
    X = (torch.rand((1, 3, 176, 176)) * 255).requires_grad_(True)
    win = MA._fspecial_gauss_1d(11, 1.5).repeat(3, 1, 1, 1).requires_grad_(True)
    for fn in (MA.ssim, MA.ms_ssim):
        with pytest.raises(NotImplementedError, match="window"):
            fn(X, X.detach(), win=win)
    with torch.no_grad():
        MA.ssim(X, X.detach(), win=win)                   # no gradient asked for: fine


def test_two_forwards_then_one_backward(MA):
    gen = torch.Generator().manual_seed(3)
    X1, X2 = (torch.rand((1, 3, 176, 176), generator=gen) * 255 for _ in range(2))
    Y = torch.rand((1, 3, 176, 176), generator=gen) * 255
    sep = []
    for Xi in (X1, X2):
        Xl = Xi.clone().requires_grad_(True)
        MA.ms_ssim(Xl, Y).backward()
        sep.append(Xl.grad)
    A, B = X1.clone().requires_grad_(True), X2.clone().requires_grad_(True)
    (MA.ms_ssim(A, Y) + MA.ms_ssim(B, Y)).backward()
    assert torch.equal(A.grad, sep[0]) and torch.equal(B.grad, sep[1])
    Z = X1.clone().requires_grad_(True)
    (MA.ms_ssim(Z, Y) + MA.ms_ssim(Z, Y)).backward()
    assert torch.equal(Z.grad, sep[0] + sep[0])
