"""Generate tests/golden/metrics.npz from the reference's unmodified src/helpers/metrics.py (a checkout named by
HIFIC_REFERENCE_ROOT) -- TEST INFRASTRUCTURE.

    HIFIC_REFERENCE_ROOT=/path/to/reference python oracle/make_golden_metrics.py

Inputs are stored as uint8 images (the data_range=1 case divides them by 255 in float32).  Outputs are the reference's,
computed on the CPU in float32 with metrics_oracle.THREADS intra-op threads; per-level (ssim, cs) come from the
reference's own _ssim and the same avg_pool2d calls as its ms_ssim loop.  The script ends by checking the oracle
restatement (oracle/metrics_oracle.py) against everything it wrote.
"""
import importlib.util
import os
import sys
import warnings

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import metrics_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "metrics.npz")


def load_reference():
    ref = os.environ.get("HIFIC_REFERENCE_ROOT", "")
    path = os.path.join(ref, "src", "helpers", "metrics.py")
    if not os.path.isfile(path):
        raise RuntimeError(f"reference metrics.py not found under HIFIC_REFERENCE_ROOT={ref!r}")
    spec = importlib.util.spec_from_file_location("reference_metrics", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def smooth_image(g, shape, lo, hi):
    """Smooth random content: a coarse random field, bilinearly upsampled, plus fine texture."""
    n, c, h, w = shape
    coarse = torch.rand((n, c, h // 8 + 2, w // 8 + 2), generator=g)
    x = F.interpolate(coarse, size=(h, w), mode="bilinear", align_corners=False)
    x = 0.8 * x + 0.2 * torch.rand(shape, generator=g)
    return (lo + (hi - lo) * x).round().clamp(0, 255).to(torch.uint8)


def perturb(g, x, sigma):
    return (x.float() + sigma * torch.randn(x.shape, generator=g)).round().clamp(0, 255).to(torch.uint8)


def inputs():
    g = torch.Generator().manual_seed(2024)
    # similar pair + unrelated (inverted) pair, odd at every level: 161 -> 81 -> 41 -> 21 -> 11, 177 -> 89 -> 45 -> 23 -> 12
    ms_x = smooth_image(g, (2, 3, 161, 177), 0, 255)
    ms_y = perturb(g, ms_x, 12.0)
    ms_y[1] = perturb(g, 255 - ms_x[1], 20.0)            # unrelated (inverted) pair: cs < 0 at every level
    sat_x = smooth_image(g, (1, 3, 161, 161), 244, 255)
    sat_y = perturb(g, sat_x, 2.0)
    small_x = smooth_image(g, (2, 3, 8, 64), 0, 255)
    small_y = perturb(g, small_x, 10.0)
    return {"ms": (ms_x, ms_y), "sat": (sat_x, sat_y), "small": (small_x, small_y)}


def ref_levels(M, X, Y, win, data_range, K, levels):
    out = []
    for level in range(levels):
        s, cs = M._ssim(X, Y, win=win, data_range=data_range, size_average=False, K=K)
        out.append((s, cs))
        if level < levels - 1:
            pad = [d % 2 for d in X.shape[2:]]
            X, Y = F.avg_pool2d(X, kernel_size=2, padding=pad), F.avg_pool2d(Y, kernel_size=2, padding=pad)
    return out


def compute(M, data):
    """Every stored output, keyed as in the npz; `data` maps case -> (X uint8, Y uint8)."""
    f = {k: (x.float(), y.float()) for k, (x, y) in data.items()}
    out = {}
    win11 = M._fspecial_gauss_1d(11, 1.5).repeat([3, 1, 1, 1])
    # MS-SSIM, default parameters, both reductions, with its per-level (ssim, cs)
    for case in ("ms", "sat"):
        X, Y = f[case]
        out[f"{case}.ms_ssim"] = M.MS_SSIM(data_range=255)(X, Y).numpy()
        out[f"{case}.ms_ssim_per_image"] = M.MS_SSIM(data_range=255, size_average=False)(X, Y).numpy()
        for l, (s, cs) in enumerate(ref_levels(M, X, Y, win11, 255, (0.01, 0.03), 5)):
            out[f"{case}.level{l}.ssim"], out[f"{case}.level{l}.cs"] = s.numpy(), cs.numpy()
    # three levels, custom weights and K, data_range 1
    X, Y = (t / 255.0 for t in f["ms"])
    w3, K3 = [0.2, 0.3, 0.5], (0.01, 0.4)
    out["custom.ms_ssim_per_image"] = M.ms_ssim(X, Y, data_range=1, size_average=False, weights=w3, K=K3).numpy()
    for l, (s, cs) in enumerate(ref_levels(M, X, Y, win11, 1, K3, 3)):
        out[f"custom.level{l}.ssim"], out[f"custom.level{l}.cs"] = s.numpy(), cs.numpy()
    # SSIM: nonnegative_ssim with both reductions, plain SSIM, SSIM(win_size=7, win_sigma=1.0)
    X, Y = f["ms"]
    out["ms.ssim_nonneg"] = M.ssim(X, Y, nonnegative_ssim=True).numpy()
    out["ms.ssim_nonneg_per_image"] = M.ssim(X, Y, nonnegative_ssim=True, size_average=False).numpy()
    for case in ("ms", "sat"):
        X, Y = f[case]
        out[f"{case}.ssim_per_image"] = M.ssim(X, Y, size_average=False).numpy()
        out[f"{case}.ssim7_per_image"] = M.SSIM(win_size=7, win_sigma=1.0, size_average=False)(X, Y).numpy()
    # SSIM on an input smaller than the window in H (smoothing along H skipped, with a warning)
    X, Y = f["small"]
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        out["small.ssim_per_image"] = M.ssim(X, Y, size_average=False).numpy()
    out["small.warning"] = np.array(str(caught[0].message))
    # PSNR of every pair (float32 arrays, as compress.py passes them), and of the data_range=1 pair
    for case, (X, Y) in f.items():
        out[f"{case}.psnr"] = M.psnr(X.numpy(), Y.numpy(), 255.)
    out["custom.psnr"] = M.psnr((f["ms"][0] / 255.0).numpy(), (f["ms"][1] / 255.0).numpy(), 1.)
    return out


def oracle_outputs(data):
    """The same outputs from oracle/metrics_oracle.py."""
    f = {k: (x.float(), y.float()) for k, (x, y) in data.items()}
    out = {}
    for case in ("ms", "sat"):
        X, Y = f[case]
        out[f"{case}.ms_ssim"] = O.ms_ssim(X, Y).numpy()
        out[f"{case}.ms_ssim_per_image"] = O.ms_ssim(X, Y, size_average=False).numpy()
        for l, (s, cs) in enumerate(O.ms_ssim_levels(X, Y, O.gauss_taps())):
            out[f"{case}.level{l}.ssim"], out[f"{case}.level{l}.cs"] = s.numpy(), cs.numpy()
    X, Y = (t / 255.0 for t in f["ms"])
    out["custom.ms_ssim_per_image"] = O.ms_ssim(X, Y, 1, False, weights=[0.2, 0.3, 0.5], K=(0.01, 0.4)).numpy()
    for l, (s, cs) in enumerate(O.ms_ssim_levels(X, Y, O.gauss_taps(), 1, (0.01, 0.4), 3)):
        out[f"custom.level{l}.ssim"], out[f"custom.level{l}.cs"] = s.numpy(), cs.numpy()
    X, Y = f["ms"]
    out["ms.ssim_nonneg"] = O.ssim(X, Y, nonnegative_ssim=True).numpy()
    out["ms.ssim_nonneg_per_image"] = O.ssim(X, Y, size_average=False, nonnegative_ssim=True).numpy()
    for case in ("ms", "sat"):
        X, Y = f[case]
        out[f"{case}.ssim_per_image"] = O.ssim(X, Y, size_average=False).numpy()
        out[f"{case}.ssim7_per_image"] = O.ssim(X, Y, size_average=False, taps=O.gauss_taps(7, 1.0)).numpy()
    X, Y = f["small"]
    out["small.ssim_per_image"] = O.ssim(X, Y, size_average=False).numpy()
    for case, (X, Y) in f.items():
        out[f"{case}.psnr"] = O.psnr(X.numpy(), Y.numpy(), 255.)
    out["custom.psnr"] = O.psnr((f["ms"][0] / 255.0).numpy(), (f["ms"][1] / 255.0).numpy(), 1.)
    return out


def main():
    torch.set_num_threads(O.THREADS)
    M = load_reference()
    data = inputs()
    out = compute(M, data)
    assert (out["ms.level0.cs"][1] < 0).all() and (out["ms.level4.cs"][1] < 0).all(), "unrelated pair: cs >= 0"
    for k, (x, y) in data.items():
        out[f"{k}.x"], out[f"{k}.y"] = x.numpy(), y.numpy()
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({os.path.getsize(OUT) / 1e6:.2f} MB, {len(out)} arrays)")
    mine = oracle_outputs(data)
    worst = 0.0
    for k, v in mine.items():
        d = float(np.max(np.abs(v.astype(np.float64) - out[k].astype(np.float64))))
        worst = max(worst, d)
        print(f"  oracle vs reference {k:32s} max |diff| {d:.3e}")
    print(f"oracle vs reference: worst {worst:.3e}")


if __name__ == "__main__":
    main()
