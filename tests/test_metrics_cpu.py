"""CPU: PSNR / SSIM / MS-SSIM (src/helpers/metrics.py) against tests/golden/metrics.npz (oracle/make_golden_metrics.py).

  * the oracle restatement (oracle/metrics_oracle.py) reproduces the reference's stored outputs bit for bit;
  * the kernels' element code (csrc/ssim_math.cuh, compiled with g++ through tests/ssim_math_host.cpp) over the whole
    golden images: pooled planes against F.avg_pool2d, per-level means and final values against the reference, and every
    valid output and pooled pixel produced by exactly one tile;
  * the host glue of hific_b200.helpers.metrics with a CPU stand-in for its two ops calls: shapes, size_average, the
    reference's validation order, exception types and messages, its warning, and the NumPy psnr path.
The kernels themselves are checked by tests/test_gpu_metrics.py on a GPU.
"""
import ctypes
import os
import subprocess
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import metrics_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "metrics.npz")
W3, K3 = [0.2, 0.3, 0.5], (0.01, 0.4)
# case -> (input key, data_range, K, weights)
MS_CASES = {"ms": ("ms", 255, (0.01, 0.03), O.DEFAULT_WEIGHTS), "sat": ("sat", 255, (0.01, 0.03), O.DEFAULT_WEIGHTS),
            "custom": ("ms", 1, K3, W3)}


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


def pair(gold, key, data_range=255):
    x, y = (torch.from_numpy(gold[f"{key}.{s}"]).float() for s in ("x", "y"))
    return (x / 255.0, y / 255.0) if data_range == 1 else (x, y)


@pytest.fixture
def oracle_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(O.THREADS)
    yield
    torch.set_num_threads(n)


def test_oracle_reproduces_the_reference_bit_for_bit(gold, oracle_threads):
    """float32 CPU convolutions sum in an order that depends on the thread count; with the generator's count the oracle
    issues the reference's exact operations and gets its exact bits."""
    for case, (key, dr, K, w) in MS_CASES.items():
        X, Y = pair(gold, key, dr)
        got = O.ms_ssim(X, Y, dr, False, weights=w, K=K).numpy()
        assert np.array_equal(got, gold[f"{case}.ms_ssim_per_image"]), case
        for l, (s, cs) in enumerate(O.ms_ssim_levels(X, Y, O.gauss_taps(), dr, K, len(w))):
            assert np.array_equal(s.numpy(), gold[f"{case}.level{l}.ssim"]), (case, l)
            assert np.array_equal(cs.numpy(), gold[f"{case}.level{l}.cs"]), (case, l)
        if case != "custom":
            assert np.array_equal(O.ms_ssim(X, Y).numpy(), gold[f"{case}.ms_ssim"])
    X, Y = pair(gold, "ms")
    assert np.array_equal(O.ssim(X, Y, nonnegative_ssim=True).numpy(), gold["ms.ssim_nonneg"])
    assert np.array_equal(O.ssim(X, Y, size_average=False, nonnegative_ssim=True).numpy(), gold["ms.ssim_nonneg_per_image"])
    for key in ("ms", "sat"):
        X, Y = pair(gold, key)
        assert np.array_equal(O.ssim(X, Y, size_average=False).numpy(), gold[f"{key}.ssim_per_image"])
        assert np.array_equal(O.ssim(X, Y, size_average=False, taps=O.gauss_taps(7, 1.0)).numpy(),
                              gold[f"{key}.ssim7_per_image"])
    X, Y = pair(gold, "small")
    assert np.array_equal(O.ssim(X, Y, size_average=False).numpy(), gold["small.ssim_per_image"])
    for key in ("ms", "sat", "small"):
        X, Y = pair(gold, key)
        assert np.array_equal(O.psnr(X.numpy(), Y.numpy()), gold[f"{key}.psnr"])


# ---------------------------------------------------------------------------------------------------------------------
# the kernels' element code on the host
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("ssim") / "ssim_math_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-x", "c++",
                    os.path.join(HERE, "ssim_math_host.cpp"), "-o", so], check=True)
    lib = ctypes.CDLL(so)
    lib.ssim_plane_value_host.restype = ctypes.c_float
    return lib


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def geom(host, h0, w0, win, level):
    out = (ctypes.c_int * 10)()
    host.ssim_level_geom_host(h0, w0, win, level, out)
    return dict(zip(("h", "w", "wh", "ww", "ho", "wo", "hp", "wp", "tiles_y", "tiles_x"), list(out)))


def host_levels(host, X, Y, taps, data_range, K, levels):
    """Runs every level like the kernels do; returns per-level (sums (planes, 2), pooled pair) and checks coverage."""
    n, c, h0, w0 = X.shape
    win = taps.numel()
    tap_table = taps.reshape(1, win).repeat(c, 1).contiguous()
    c1, c2 = ctypes.c_float((K[0] * data_range) ** 2), ctypes.c_float((K[1] * data_range) ** 2)
    x, y = X.contiguous(), Y.contiguous()
    out = []
    for level in range(levels):
        g = geom(host, h0, w0, win, level)
        assert (g["h"], g["w"]) == tuple(x.shape[2:])
        tiles = g["tiles_y"] * g["tiles_x"]
        partials = torch.zeros((n * c, tiles, 2), dtype=torch.float64)
        out_cover = torch.zeros((n * c, g["ho"], g["wo"]), dtype=torch.int32)
        pool_cover = torch.zeros((n * c, g["hp"], g["wp"]), dtype=torch.int32)
        last = level == levels - 1
        px = None if last else torch.empty((n, c, g["hp"], g["wp"]))
        py = None if last else torch.empty_like(px)
        host.ssim_level_host(_p(x), _p(y), n * c, c, h0, w0, level, _p(tap_table), win, c1, c2,
                             _p(px) if px is not None else None, _p(py) if py is not None else None, _p(partials),
                             _p(out_cover), _p(pool_cover))
        assert bool((out_cover == 1).all()), ("valid outputs not covered exactly once", level)
        if not last:
            assert bool((pool_cover == 1).all()), ("pooled pixels not owned exactly once", level)
        out.append((partials.sum(1), g, (px, py), (x, y)))
        x, y = px, py
    return out


def assert_within_ulp(got, want, ulps=1):
    spacing = np.spacing(np.abs(want.numpy()).astype(np.float32))
    assert bool(np.all(np.abs(got.numpy() - want.numpy()) <= ulps * spacing))


@pytest.mark.parametrize("case", sorted(MS_CASES))
def test_kernel_element_code_on_golden_images(host, gold, case):
    key, dr, K, weights = MS_CASES[case]
    X, Y = pair(gold, key, dr)
    n, c = X.shape[:2]
    levels = host_levels(host, X, Y, O.gauss_taps(), dr, K, len(weights))
    sums_all = []
    for l, (sums, g, (px, py), (x, y)) in enumerate(levels):
        count = g["ho"] * g["wo"]
        means = (sums / count).float().reshape(n, c, 2)
        assert np.abs(means[..., 0].numpy() - gold[f"{case}.level{l}.ssim"]).max() < 1e-6, (case, l)
        assert np.abs(means[..., 1].numpy() - gold[f"{case}.level{l}.cs"]).max() < 1e-6, (case, l)
        if px is not None:
            pad = [s % 2 for s in x.shape[2:]]
            assert_within_ulp(px, F.avg_pool2d(x, 2, padding=pad))
            assert_within_ulp(py, F.avg_pool2d(y, 2, padding=pad))
        sums_all.append(sums)
    per_plane = torch.stack(sums_all, 1).contiguous()           # (planes, levels, 2)
    wts = (ctypes.c_float * len(weights))(*weights)
    vals = torch.tensor([host.ssim_plane_value_host(_p(per_plane[p]), wts, len(weights), X.shape[2], X.shape[3], 11, 1)
                         for p in range(n * c)], dtype=torch.float64).reshape(n, c)
    assert np.abs(vals.mean(1).numpy() - gold[f"{case}.ms_ssim_per_image"]).max() < 1e-6
    if case != "custom":
        assert abs(vals.mean().item() - float(gold[f"{case}.ms_ssim"])) < 1e-6


@pytest.mark.parametrize("case,win,sigma", [("ms", 7, 1.0), ("sat", 7, 1.0), ("small", 11, 1.5), ("ms", 11, 1.5)])
def test_kernel_element_code_single_level(host, gold, case, win, sigma):
    """ssim(): one level, the finalisation's weight-1 path; `small` is shorter than the window in H (not smoothed)."""
    X, Y = pair(gold, case)
    n, c = X.shape[:2]
    (sums, g, _, _), = host_levels(host, X, Y, O.gauss_taps(win, sigma), 255, (0.01, 0.03), 1)
    if case == "small":
        assert g["wh"] == 1 and g["ho"] == X.shape[2]
    one = (ctypes.c_float * 1)(1.0)
    for relu_last, key in ((0, "ssim_per_image"), (1, "ssim_nonneg_per_image")):
        if relu_last and (case != "ms" or win != 11):
            continue
        vals = torch.tensor([host.ssim_plane_value_host(_p(sums[p].contiguous()), one, 1, X.shape[2], X.shape[3], win,
                                                        relu_last) for p in range(n * c)], dtype=torch.float64)
        want = gold[f"{case}.{'ssim7_per_image' if win == 7 else key}"]
        assert np.abs(vals.reshape(n, c).mean(1).numpy() - want).max() < 1e-6


def test_tiles_cover_odd_sizes_exactly_once(host):
    """Ownership on sizes odd at several levels, and where the pooled grid needs more tiles than the output grid."""
    g = torch.Generator().manual_seed(5)
    for h, w, win in ((177, 243, 11), (165, 263, 11), (97, 161, 3), (35, 31, 31), (64, 64, 11), (1, 1, 1)):
        X = torch.rand((1, 2, h, w), generator=g) * 255
        Y = torch.rand((1, 2, h, w), generator=g) * 255
        host_levels(host, X, Y, O.gauss_taps(win, 1.5), 255, (0.01, 0.03), 3)


# ---------------------------------------------------------------------------------------------------------------------
# host glue of hific_b200.helpers.metrics, with a CPU stand-in for ops
# ---------------------------------------------------------------------------------------------------------------------
class CpuOps:
    """Stand-in for the two ops calls of helpers/metrics.py, computed with the oracle's float32 operations on the CPU."""

    def __init__(self):
        self.calls = []

    def ssim_levels(self, x, y, taps, c1, c2, weights, relu_last, size_average):
        self.calls.append(("ssim_levels", tuple(x.shape), taps.clone(), c1, c2, list(weights), relu_last, size_average))
        vals = None
        for level, w in enumerate(weights):
            t = taps[0]
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
            x, y = O.pool(x), O.pool(y)
        return vals.mean() if size_average else vals.mean(1)

    def psnr(self, a, b, max_val):
        self.calls.append(("psnr",))
        return torch.from_numpy(O.psnr(a, b, max_val))


@pytest.fixture
def M(monkeypatch):
    from hific_b200.helpers import metrics
    fake = CpuOps()
    monkeypatch.setattr(metrics, "ops", fake)
    monkeypatch.setattr(metrics, "_require_cuda", lambda X, Y, what: None)
    metrics.fake = fake
    return metrics


def test_public_names():
    from hific_b200.helpers import metrics
    for name in ("psnr", "ssim", "ms_ssim", "SSIM", "MS_SSIM", "_fspecial_gauss_1d"):
        assert hasattr(metrics, name)
    g = metrics._fspecial_gauss_1d(11, 1.5)
    assert g.shape == (1, 1, 11) and g.dtype == torch.float32
    assert torch.equal(g.reshape(-1), O.gauss_taps(11, 1.5))
    assert metrics.SSIM(channel=3).win.shape == (3, 1, 1, 11) and metrics.MS_SSIM(channel=4).win.shape == (4, 1, 1, 11)


def test_shapes_and_size_average(M):
    X = torch.rand((2, 3, 176, 180)) * 255
    Y = (X + torch.randn(X.shape) * 5).clamp(0, 255)
    assert M.ms_ssim(X, Y).shape == () and M.ms_ssim(X, Y, size_average=False).shape == (2,)
    assert M.ssim(X, Y).shape == () and M.ssim(X, Y, size_average=False).shape == (2,)
    assert M.MS_SSIM(data_range=255)(X, Y).shape == () and M.SSIM(size_average=False)(X, Y).shape == (2,)
    per = M.ms_ssim(X, Y, size_average=False)
    assert torch.allclose(per.mean(), M.ms_ssim(X, Y), atol=1e-7)
    # what reaches the kernels: default weights (fp32-rounded), constants, relu flags, a (C, win) tap table
    M.fake.calls.clear()
    M.ms_ssim(X, Y, data_range=1, K=(0.02, 0.4), weights=[0.5, 0.5])
    _, shape, taps, c1, c2, w, relu_last, avg = M.fake.calls[-1]
    assert shape == (2, 3, 176, 180) and taps.shape == (3, 11) and w == [0.5, 0.5] and relu_last and avg
    assert c1 == pytest.approx(0.02 ** 2) and c2 == pytest.approx(0.4 ** 2)
    M.ms_ssim(X, Y)
    assert M.fake.calls[-1][5] == [float(np.float32(v)) for v in O.DEFAULT_WEIGHTS]
    M.ssim(X, Y, nonnegative_ssim=True, win_size=7, win_sigma=1.0)
    _, _, taps, _, _, w, relu_last, _ = M.fake.calls[-1]
    assert w == [1.0] and relu_last and torch.equal(taps[1], O.gauss_taps(7, 1.0))
    # `win` overrides win_size, per channel
    win = torch.stack([O.gauss_taps(5, 1.0), O.gauss_taps(5, 2.0), O.gauss_taps(5, 3.0)]).reshape(3, 1, 1, 5)
    M.ssim(X, Y, win=win, win_size=11)
    assert torch.equal(M.fake.calls[-1][2], win.reshape(3, 5))
    # trailing singleton dimensions are squeezed
    assert M.ssim(X[..., None], Y[..., None], size_average=False).shape == (2,)


def test_golden_values_through_the_glue(M, gold, oracle_threads):
    X, Y = pair(gold, "ms")
    assert np.array_equal(M.ms_ssim(X, Y, size_average=False).numpy(), gold["ms.ms_ssim_per_image"])
    assert np.array_equal(M.SSIM(win_size=7, win_sigma=1.0, size_average=False)(X, Y).numpy(), gold["ms.ssim7_per_image"])
    assert np.array_equal(M.ssim(X, Y, nonnegative_ssim=True, size_average=False).numpy(), gold["ms.ssim_nonneg_per_image"])


def test_validation_matches_the_reference(M):
    X = torch.rand((1, 3, 176, 176))
    with pytest.raises(ValueError, match="^Input images should have the same dimensions.$"):
        M.ssim(X, X[:, :2])
    with pytest.raises(ValueError, match="^Input images should have the same dimensions.$"):
        M.ms_ssim(X, X[:, :2])
    bad = torch.rand((3, 176, 176))
    for fn in (M.ssim, M.ms_ssim):
        with pytest.raises(ValueError, match=r"^Input images should be 4-d or 5-d tensors, but got torch.Size\(\[3, 176, "
                                             r"176\]\)$"):
            fn(bad, bad)
        with pytest.raises(ValueError, match="^Input images should have the same dtype.$"):
            fn(X, X.double())
        with pytest.raises(ValueError, match="^Window size should be odd.$"):
            fn(X, X, win_size=10)
        with pytest.raises(ValueError, match="^Window size should be odd.$"):
            fn(X, X, win=torch.ones(3, 1, 1, 4))
    # ms_ssim checks the dtype before the number of dimensions, ssim after
    with pytest.raises(ValueError, match="same dtype"):
        M.ms_ssim(bad, bad.double())
    with pytest.raises(ValueError, match="4-d or 5-d"):
        M.ssim(bad, bad.double())
    small = torch.rand((1, 3, 160, 200))
    with pytest.raises(AssertionError, match="^Image size should be larger than 160 due to the 4 downsamplings in "
                                             "ms-ssim$"):
        M.ms_ssim(small, small)
    with pytest.raises(AssertionError, match="larger than 96 "):
        M.ms_ssim(torch.rand((1, 3, 96, 200)), torch.rand((1, 3, 96, 200)), win_size=7)


def test_unsupported_inputs_raise(M, monkeypatch):
    X = torch.rand((1, 3, 176, 176))
    for fn in (M.ssim, M.ms_ssim):
        with pytest.raises(NotImplementedError, match="float32"):
            fn(X.double(), X.double())
        with pytest.raises(NotImplementedError, match="5-d"):
            fn(torch.rand((1, 3, 4, 176, 176)), torch.rand((1, 3, 4, 176, 176)))
        with pytest.raises(NotImplementedError, match="window size 33"):
            fn(torch.rand((1, 3, 600, 600)), torch.rand((1, 3, 600, 600)), win_size=33)
        with pytest.raises(NotImplementedError, match="forward only"):
            fn(X.clone().requires_grad_(True), X)
        with torch.no_grad():
            fn(X.clone().requires_grad_(True), X)           # no gradient asked for: fine
    with pytest.raises(NotImplementedError, match="at most 8 levels"):
        M.ms_ssim(X, X, weights=[0.1] * 9)
    from hific_b200.helpers import metrics
    monkeypatch.undo()
    for fn in (metrics.ssim, metrics.ms_ssim):
        with pytest.raises(RuntimeError, match="CUDA tensors"):
            fn(X, X)
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        metrics.psnr(X, X)


def test_warning_matches_the_reference(M, gold):
    X, Y = pair(gold, "small")
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        M.ssim(X, Y, size_average=False)
    assert [str(w.message) for w in caught] == [str(gold["small.warning"])]
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        M.ssim(*pair(gold, "ms"))


def test_numpy_psnr_is_the_reference_bit_for_bit(gold):
    from hific_b200.helpers import metrics
    for key in ("ms", "sat", "small"):
        x, y = (gold[f"{key}.{s}"].astype(np.float32) for s in ("x", "y"))
        got = metrics.psnr(x, y, 255.)
        assert got.dtype == np.float64 and np.array_equal(got, gold[f"{key}.psnr"])
    x, y = (gold[f"ms.{s}"].astype(np.float32) for s in ("x", "y"))
    got = metrics.psnr((torch.from_numpy(x) / 255.0).numpy(), (torch.from_numpy(y) / 255.0).numpy(), 1.)
    assert np.array_equal(got, gold["custom.psnr"])
