"""Per-call time of PSNR / SSIM / MS-SSIM (hific_b200.helpers.metrics, csrc/ssim.cu) against the reference formulation,
and compress.py's per-batch loop body with either metrics path.  One GPU process; prints and writes one JSON document.

    python tools/metrics_bench.py --out profiles/r03_metrics_bench.json

Per shape (1x3x512x768, 1x3x1365x2048, 8x3x1024x1024; every shape warmed first), CUDA events around each call:
  (a) the reference formulation run eagerly on the GPU (oracle/metrics_oracle.py: the reference's F.conv2d / avg_pool2d
      calls, float32, torch's default TF32 settings),
  (b) the new kernels,
  (c) for PSNR, the reference path: device-to-host copy of both images plus NumPy float64.
Achieved bandwidth uses the algorithmic bytes: per level, X and Y read once and the pooled pair written.
The loop body (compress, decompress, LPIPS, PSNR, MS-SSIM at 1x3x512x768) runs random-init weights: the latents are not
those of a trained model, which changes the rate and therefore the host coder's time.
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("HFC_LPIPS_SYNTHETIC", "1")

from hific_b200 import synth  # noqa: E402
from hific_b200.helpers import metrics as M  # noqa: E402
from oracle import metrics_oracle as O  # noqa: E402

SHAPES = [(1, 3, 512, 768), (1, 3, 1365, 2048), (8, 3, 1024, 1024)]
HBM_PEAK = 7.7e12          # B/s, HGX B200 data sheet, one GPU
L2_BYTES = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def ms_ssim_bytes(shape, levels=5):
    n, c, h, w = shape
    total = 0
    for level in range(levels):
        total += 2 * n * c * h * w * 4
        h, w = (h + 1) // 2, (w + 1) // 2
        if level < levels - 1:
            total += 2 * n * c * h * w * 4
    return total


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


def time_host(fn, reps):
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": float(np.median(times)), "min_ms": float(np.min(times)), "reps": reps}


def pair(shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n, c, h, w = shape
    x = torch.rand((n, c, h // 16 + 1, w // 16 + 1), device="cuda", generator=g) * 255
    x = torch.nn.functional.interpolate(x, size=(h, w), mode="bilinear", align_corners=False)
    x = (x + 20 * torch.rand(shape, device="cuda", generator=g)).clamp(0, 255).contiguous()
    y = (x + 8 * torch.randn(shape, device="cuda", generator=g)).clamp(0, 255).contiguous()
    return x, y


def per_call(reps):
    mod_new = M.MS_SSIM(data_range=255)
    inputs = {s: pair(s, sum(s)) for s in SHAPES}
    for x, y in inputs.values():                         # warm every shape and path
        for _ in range(3):
            O.ms_ssim(x, y), mod_new(x, y), M.psnr(x, y), M.ssim(x, y), O.ssim(x, y)
            M.psnr(x.cpu().numpy(), y.cpu().numpy())
    torch.cuda.synchronize()
    rows = []
    for shape, (x, y) in inputs.items():
        r = {"shape": list(shape)}
        r["ms_ssim_reference_eager_ms"] = time_cuda(lambda: O.ms_ssim(x, y), reps)
        r["ms_ssim_kernels_ms"] = time_cuda(lambda: mod_new(x, y), reps)
        r["ssim_reference_eager_ms"] = time_cuda(lambda: O.ssim(x, y), reps)
        r["ssim_kernels_ms"] = time_cuda(lambda: M.ssim(x, y), reps)
        r["psnr_kernels_ms"] = time_cuda(lambda: M.psnr(x, y), reps)
        r["psnr_reference_d2h_numpy_ms"] = time_host(lambda: M.psnr(x.cpu().numpy(), y.cpu().numpy()), max(3, reps // 4))
        r["agreement"] = {
            "ms_ssim_kernels_minus_eager_tf32": float((mod_new(x, y) - O.ms_ssim(x, y)).abs()),
            "ms_ssim_kernels_minus_fp64_oracle": float((mod_new(x, y).double()
                                                        - O.ms_ssim(x, y, dtype=torch.float64)).abs()),
            "psnr_kernels_minus_numpy_db": float(np.max(np.abs(M.psnr(x, y).cpu().numpy()
                                                               - M.psnr(x.cpu().numpy(), y.cpu().numpy())))),
        }
        b = ms_ssim_bytes(shape)
        t = r["ms_ssim_kernels_ms"]["median_ms"] * 1e-3
        r["ms_ssim_algorithmic_bytes"] = b
        r["ms_ssim_kernels_GBps"] = b / t / 1e9
        r["ms_ssim_kernels_fraction_of_hbm_peak"] = b / t / HBM_PEAK
        pb = 2 * x.numel() * 4
        r["psnr_kernels_GBps"] = pb / (r["psnr_kernels_ms"]["median_ms"] * 1e-3) / 1e9
        r["psnr_kernels_fraction_of_hbm_peak"] = r["psnr_kernels_GBps"] * 1e9 / HBM_PEAK
        r["inputs_bytes"] = pb
        r["inputs_fit_in_l2"] = pb < L2_BYTES
        rows.append(r)
        print(json.dumps(r), flush=True)
    return rows


def loop_body(reps):
    """compress.py:147-173 at 1x3x512x768: compress, decompress, LPIPS, PSNR, MS-SSIM."""
    from hific_b200.config import ModelModes, mse_lpips_args
    from hific_b200.loss.perceptual import PerceptualLoss
    from hific_b200.model import Model
    gold = np.load(os.path.join(ROOT, "tests", "golden", "entropy_coding.npz"))
    m = Model(mse_lpips_args(), logging.getLogger("bench"), model_mode=ModelModes.EVALUATION)
    m.load_state_dict(synth.synth_state_dict(0), strict=False)
    m.Hyperprior.hyperprior_entropy_model._register_tables(gold["hyper.CDF"], gold["hyper.CDF_offset"],
                                                           gold["hyper.CDF_length"])
    m = m.cuda().eval()
    lpips = PerceptualLoss(model="net-lin", net="alex", use_gpu=True).cuda()
    x = synth.synth_image(1, 512, 768, 3).cuda()
    ref_ms = M.MS_SSIM(data_range=255)

    def body(new):
        with torch.no_grad():
            co = m.compress(x, silent=True)
            rec = m.decompress(co)
            lp = lpips.forward(rec, x, normalize=True)
            if new:
                ps = M.psnr(rec * 255.0, x * 255.0, 255.0)
                ms = ref_ms(rec * 255.0, x * 255.0)
            else:
                ps = M.psnr(rec.cpu().numpy() * 255.0, x.cpu().numpy() * 255.0, 255.0)
                ms = O.ms_ssim(rec * 255.0, x * 255.0)
            return lp, ps, ms

    for new in (False, True, False, True):
        body(new)
    out = {}
    for new, tag in ((False, "reference_metrics"), (True, "kernel_metrics")):
        t = time_host(lambda: body(new), reps)
        out[tag] = {"per_image_ms": t, "images_per_s": 1e3 / t["median_ms"]}
    out["note"] = "random-init weights: the rate, and with it the host coder's time, are not a trained model's"
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="where to write the JSON document")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--loop-reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_bench needs a CUDA device")
    doc = {"card": card(), "allow_tf32": {"cudnn": torch.backends.cudnn.allow_tf32,
                                          "matmul": torch.backends.cuda.matmul.allow_tf32},
           "per_call": per_call(a.reps), "loop_body_1x3x512x768": loop_body(a.loop_reps)}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc["card"]))


if __name__ == "__main__":
    main()
