"""Generate tests/golden/noise_generator_ls_gan.npz from two functions of the REAL reference -- TEST INFRASTRUCTURE, needs a
checkout of the reference (HIFIC_REFERENCE_ROOT, see oracle/ref_shim.py).

    HIFIC_REFERENCE_ROOT=<checkout> python oracle/make_golden_noise_gan.py

  * `gan_loss('least_squares', ...)` (src/loss/losses.py:43-66): value and gradients w.r.t. both logit tensors, in
    generator and discriminator mode, on the seeded logits of tests/test_gan_loss_variants_cpu.py (`_disc_out(2)`);
  * the `sample_noise=True` Generator (src/network/generator.py:105-107, 149-161) built under torch.manual_seed(9): its
    output on a seeded y_hat with a fixed noise draw.  Its 43 M weights are NOT stored: the product's mirror module draws
    them bit for bit under the same seed; the names, shapes and float64 sums of the reference's tensors are stored so the
    test can check that.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402


def disc_logits(seed):
    """The logits of tests/test_gan_loss_variants_cpu.py: `_disc_out(seed)`."""
    g = torch.Generator().manual_seed(seed)
    lr = torch.randn((2 * 256, 1), generator=g).requires_grad_(True)
    lg = torch.randn((2 * 256, 1), generator=g).requires_grad_(True)
    return lr, lg


def noise_generator_inputs():
    g = torch.Generator().manual_seed(10)
    y_hat = torch.round(torch.randn((2, 220, 8, 8), generator=g) * 2)
    z = torch.randn((2, 32, 8, 8), generator=g)
    return y_hat, z


def main():
    ref_shim.install()
    from collections import namedtuple
    from src.loss import losses as R
    import src.network.generator as ref_generator
    Disc_out = namedtuple("Disc_out", ["D_real", "D_gen", "D_real_logits", "D_gen_logits"])
    out = {}
    for mode in ("generator_loss", "discriminator_loss"):
        lr, lg = disc_logits(2)
        loss = R.gan_loss("least_squares", Disc_out(torch.sigmoid(lr), torch.sigmoid(lg), lr, lg), mode)
        loss.backward()
        out[f"ls_gan.{mode}.loss"] = loss.detach().numpy()
        out[f"ls_gan.{mode}.grad_gen"] = lg.grad.numpy()
        out[f"ls_gan.{mode}.has_grad_real"] = np.array(lr.grad is not None)
        if lr.grad is not None:
            out[f"ls_gan.{mode}.grad_real"] = lr.grad.numpy()

    torch.manual_seed(9)
    ref = ref_generator.Generator((220, 8, 8), 2, C=220, n_residual_blocks=2, sample_noise=True, noise_dim=32)
    sd = ref.state_dict()
    out["noise_generator.keys"] = np.array(list(sd))
    out["noise_generator.shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
    out["noise_generator.sums"] = np.array([float(v.double().sum()) for v in sd.values()])
    y_hat, z = noise_generator_inputs()
    orig = torch.randn
    torch.randn = lambda *a, **k: z.clone()
    try:
        with torch.no_grad():
            out["noise_generator.output"] = ref(y_hat).numpy()
    finally:
        torch.randn = orig
    path = os.path.join(ROOT, "tests", "golden", "noise_generator_ls_gan.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
