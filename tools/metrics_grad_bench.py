"""Forward + backward time of MS_SSIM / SSIM with gradients (hific_b200.helpers.metrics_autograd, csrc/ssim.cu) against
eager autograd of the reference formulation on the same GPU.  One GPU process; prints and writes one JSON document.

    python tools/metrics_grad_bench.py --out profiles/r04_metrics_grad_bench.json

Per shape (1x3x512x768, 1x3x1365x2048, 8x3x1024x1024; every shape and path warmed first), CUDA events around one
`loss = 1 - metric(X, Y); loss.backward()` with X requiring a gradient (the training case: X is the reconstruction, Y the
target):
  (a) the reference formulation under eager autograd (oracle/metrics_oracle.py: the reference's F.conv2d / avg_pool2d
      calls in float32 with torch's default settings, i.e. TF32 convolutions where cuDNN picks them),
  (b) the kernels: levels + 1 forward launches, 2 * levels + 1 backward launches.
At 8x3x1024x1024 the two inputs are 201 MB, larger than the 126 MB L2.  Achieved bandwidth uses the algorithmic bytes:
forward, per level X and Y read and the pooled pair written; backward, per level X and Y read twice, the four fp32
gradient maps written and read once (16 B per valid output each way), the next level's dX read and dX written.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hific_b200.helpers import metrics_autograd as MA  # noqa: E402
from oracle import metrics_oracle as O  # noqa: E402

SHAPES = [(1, 3, 512, 768), (1, 3, 1365, 2048), (8, 3, 1024, 1024)]
HBM_PEAK = 7.7e12          # B/s, HGX B200 data sheet, one GPU
L2_BYTES = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def fwd_bwd_bytes(shape, levels, win=11):
    """Algorithmic bytes of the kernels' forward + backward with one input needing a gradient."""
    n, c, h, w = shape
    planes = n * c
    fwd = bwd = 0
    for level in range(levels):
        px = planes * h * w
        wh, ww = (win if h >= win else 1), (win if w >= win else 1)
        outs = planes * (h - wh + 1) * (w - ww + 1)
        hp, wp = (h + 1) // 2, (w + 1) // 2
        last = level == levels - 1
        fwd += 2 * px * 4 + (0 if last else 2 * planes * hp * wp * 4)
        bwd += 2 * px * 4 + outs * 16                                  # grad maps: X, Y in, maps out
        bwd += outs * 16 + 2 * px * 4 + px * 4                         # level backward: maps, X, Y in, dX out
        bwd += 0 if last else planes * hp * wp * 4                     # the next level's dX
        h, w = hp, wp
    return fwd, bwd


def time_cuda(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        start.record()
        fn()
        end.record()
        end.synchronize()
        times.append(start.elapsed_time(end))
    return {"median_ms": float(np.median(times)), "min_ms": float(np.min(times)), "reps": reps}


def pair(shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n, c, h, w = shape
    x = torch.rand((n, c, h // 16 + 1, w // 16 + 1), device="cuda", generator=g) * 255
    x = torch.nn.functional.interpolate(x, size=(h, w), mode="bilinear", align_corners=False)
    x = (x + 20 * torch.rand(shape, device="cuda", generator=g)).clamp(0, 255).contiguous()
    y = (x + 8 * torch.randn(shape, device="cuda", generator=g)).clamp(0, 255).contiguous()
    return x, y


def step(metric, xl, y):
    xl.grad = None
    (1 - metric(xl, y)).backward()


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def per_call(reps):
    kernels = {"ms_ssim": MA.MS_SSIM(data_range=255), "ssim": MA.SSIM(data_range=255)}
    eager = {"ms_ssim": lambda a, b: O.ms_ssim(a, b), "ssim": lambda a, b: O.ssim(a, b)}
    inputs = {s: pair(s, sum(s)) for s in SHAPES}
    leaves = {s: x.clone().requires_grad_(True) for s, (x, _) in inputs.items()}
    for s, (_, y) in inputs.items():                    # warm every shape and path
        for _ in range(3):
            for name in kernels:
                step(kernels[name], leaves[s], y)
                step(eager[name], leaves[s], y)
    torch.cuda.synchronize()
    rows = []
    for shape, (x, y) in inputs.items():
        xl = leaves[shape]
        r = {"shape": list(shape), "inputs_bytes": 2 * x.numel() * 4, "inputs_fit_in_l2": 2 * x.numel() * 4 < L2_BYTES}
        for name, levels in (("ms_ssim", 5), ("ssim", 1)):
            r[f"{name}_fwd_bwd_reference_eager_autograd_ms"] = time_cuda(lambda: step(eager[name], xl, y), reps)
            r[f"{name}_fwd_bwd_kernels_ms"] = time_cuda(lambda: step(kernels[name], xl, y), reps)
            r[f"{name}_fwd_kernels_ms"] = time_cuda(lambda: kernels[name](x, y), reps)
            tk = r[f"{name}_fwd_bwd_kernels_ms"]["median_ms"]
            te = r[f"{name}_fwd_bwd_reference_eager_autograd_ms"]["median_ms"]
            r[f"{name}_speedup_vs_eager"] = te / tk
            r[f"{name}_kernels_beat_eager"] = tk < te
            fb, bb = fwd_bwd_bytes(shape, levels)
            r[f"{name}_algorithmic_bytes"] = {"forward": fb, "backward": bb}
            r[f"{name}_fwd_bwd_kernels_GBps"] = (fb + bb) / (tk * 1e-3) / 1e9
            r[f"{name}_fwd_bwd_kernels_fraction_of_hbm_peak"] = (fb + bb) / (tk * 1e-3) / HBM_PEAK
            step(kernels[name], xl, y)
            gk = xl.grad.clone()
            step(eager[name], xl, y)
            ge = xl.grad.clone()
            x64 = x.double().requires_grad_(True)
            fn64 = O.ms_ssim if name == "ms_ssim" else O.ssim
            (1 - fn64(x64, y.double(), dtype=torch.float64)).backward()
            r[f"{name}_agreement"] = {"kernels_grad_rel_l2_vs_fp64": rel_l2(gk, x64.grad),
                                      "eager_default_grad_rel_l2_vs_fp64": rel_l2(ge, x64.grad)}
            del x64
        rows.append(r)
        print(json.dumps(r), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="where to write the JSON document")
    ap.add_argument("--reps", type=int, default=30)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_grad_bench needs a CUDA device")
    doc = {"card": card(), "allow_tf32": {"cudnn": torch.backends.cudnn.allow_tf32,
                                          "matmul": torch.backends.cuda.matmul.allow_tf32},
           "note": "eager = the reference formulation under torch autograd with torch's defaults (TF32 convolutions); "
                   "X requires a gradient, Y does not",
           "per_call": per_call(a.reps)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc["card"]))


if __name__ == "__main__":
    main()
