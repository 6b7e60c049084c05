"""Generate tests/golden/metrics_grad.npz: gradients of the reference's unmodified src/helpers/metrics.py (a checkout named
by HIFIC_REFERENCE_ROOT) with respect to both images -- TEST INFRASTRUCTURE.

    HIFIC_REFERENCE_ROOT=/path/to/reference python oracle/make_golden_metrics_grad.py

The inputs are the uint8 images already stored in tests/golden/metrics.npz.  Each case runs the reference's ms_ssim /
ssim under autograd, in float32 on the CPU with metrics_oracle.THREADS intra-op threads, and back-propagates a loss
(the value itself when size-averaged, else the sum of the per-image values).  Full gradients would not fit a small test
vector, so every case stores a seeded sample of elements (`{case}.idx` into the flattened tensor; SAMPLE_LARGE of them
for the default MS-SSIM of `ms` and `sat`, SAMPLE elsewhere) and the per-image float64 sums of squares of the whole dX
and dY (`{case}.dX_sumsq`, shape (N,)), which are exactly 0 for the inverted pair of `ms`.  The script ends by checking
oracle/metrics_oracle.py's autograd against everything it wrote.
"""
import importlib.util
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import metrics_oracle as O  # noqa: E402

SRC = os.path.join(ROOT, "tests", "golden", "metrics.npz")
OUT = os.path.join(ROOT, "tests", "golden", "metrics_grad.npz")
SAMPLE = 512
SAMPLE_LARGE = 2048
W3, K3 = [0.2, 0.3, 0.5], (0.01, 0.4)
LARGE = ("ms", "sat")


def load_reference():
    ref = os.environ.get("HIFIC_REFERENCE_ROOT", "")
    path = os.path.join(ref, "src", "helpers", "metrics.py")
    if not os.path.isfile(path):
        raise RuntimeError(f"reference metrics.py not found under HIFIC_REFERENCE_ROOT={ref!r}")
    spec = importlib.util.spec_from_file_location("reference_metrics", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cases(M):
    """case -> (input key, scale, loss(X, Y)) with M = the reference module or the oracle adapter below."""
    return {
        "ms": ("ms", 1.0, lambda X, Y: M.ms_ssim(X, Y, data_range=255)),
        "sat": ("sat", 1.0, lambda X, Y: M.ms_ssim(X, Y, data_range=255)),
        "custom": ("ms", 1 / 255.0, lambda X, Y: M.ms_ssim(X, Y, data_range=1, size_average=False, weights=W3,
                                                            K=K3).sum()),
        "ssim": ("ms", 1.0, lambda X, Y: M.ssim(X, Y, data_range=255, size_average=False).sum()),
        "ssim_nonneg": ("ms", 1.0, lambda X, Y: M.ssim(X, Y, data_range=255, nonnegative_ssim=True)),
        "ssim7": ("ms", 1.0, lambda X, Y: M.ssim(X, Y, data_range=255, win_size=7, win_sigma=1.0)),
        "small": ("small", 1.0, lambda X, Y: M.ssim(X, Y, data_range=255, size_average=False).sum()),
    }


class OracleAdapter:
    """The reference's ms_ssim / ssim signatures over oracle/metrics_oracle.py, for any dtype."""

    def __init__(self, dtype=torch.float32):
        self.dtype = dtype

    def ms_ssim(self, X, Y, data_range=255, size_average=True, weights=None, K=(0.01, 0.03)):
        return O.ms_ssim(X, Y, data_range, size_average, weights=weights, K=K, dtype=self.dtype)

    def ssim(self, X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, K=(0.01, 0.03),
             nonnegative_ssim=False):
        return O.ssim(X, Y, data_range, size_average, taps=O.gauss_taps(win_size, win_sigma), K=K,
                      nonnegative_ssim=nonnegative_ssim, dtype=self.dtype)


def inputs(src, key, scale):
    x, y = (torch.from_numpy(src[f"{key}.{s}"]).float() for s in ("x", "y"))
    return (x * scale, y * scale) if scale != 1.0 else (x, y)


def grads(M, src, case, dtype=torch.float32):
    key, scale, loss = cases(M)[case]
    X, Y = inputs(src, key, scale)
    X, Y = X.to(dtype).requires_grad_(True), Y.to(dtype).requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        loss(X, Y).backward()
    return X.grad, Y.grad


def sample_index(numel, case):
    g = torch.Generator().manual_seed(sum(map(ord, case)))
    return torch.randperm(numel, generator=g)[:SAMPLE_LARGE if case in LARGE else SAMPLE].to(torch.int32)


def per_image_sumsq(g):
    return (g.double() ** 2).flatten(1).sum(1)


def main():
    torch.set_num_threads(O.THREADS)
    M = load_reference()
    src = np.load(SRC)
    out = {}
    for case in cases(M):
        dX, dY = grads(M, src, case)
        assert torch.isfinite(dX).all() and torch.isfinite(dY).all(), case
        idx = sample_index(dX.numel(), case)
        out[f"{case}.idx"] = idx.numpy()
        for name, g in (("dX", dX), ("dY", dY)):
            out[f"{case}.{name}_sample"] = g.reshape(-1)[idx.long()].numpy()
            out[f"{case}.{name}_sumsq"] = per_image_sumsq(g).numpy()
    assert out["ms.dX_sumsq"][1] == 0 and out["ms.dY_sumsq"][1] == 0, "inverted pair: gradient not exactly 0"
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({os.path.getsize(OUT) / 1e6:.3f} MB, {len(out)} arrays)")
    A = OracleAdapter()
    for case in cases(M):
        dX, dY = grads(A, src, case)
        idx = torch.from_numpy(out[f"{case}.idx"]).long()
        same = all(np.array_equal(g.reshape(-1)[idx].numpy(), out[f"{case}.{name}_sample"])
                   and np.array_equal(per_image_sumsq(g).numpy(), out[f"{case}.{name}_sumsq"])
                   for name, g in (("dX", dX), ("dY", dY)))
        print(f"  oracle autograd vs reference {case:12s} bit-identical: {same}")


if __name__ == "__main__":
    main()
