"""CPU: the least-squares GAN loss variant (`gan_loss_type='least_squares'`, src/loss/losses.py:43-50, 52-66) of
hific_b200.loss.losses.gan_loss -- values and gradients against the formulas of the reference, and against what the reference's
own function computed (tests/golden/noise_generator_ls_gan.npz, oracle/make_golden_noise_gan.py)."""
import os
from collections import namedtuple

import numpy as np
import pytest
import torch

from hific_b200.loss import losses as L

Disc_out = namedtuple("Disc_out", ["D_real", "D_gen", "D_real_logits", "D_gen_logits"])
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "noise_generator_ls_gan.npz")


def _disc_out(seed):
    g = torch.Generator().manual_seed(seed)
    lr = torch.randn((2 * 256, 1), generator=g).requires_grad_(True)
    lg = torch.randn((2 * 256, 1), generator=g).requires_grad_(True)
    return Disc_out(torch.sigmoid(lr), torch.sigmoid(lg), lr, lg), lr, lg


@pytest.mark.parametrize("mode", ["generator_loss", "discriminator_loss"])
def test_least_squares_gan_loss_formula(mode):
    out, lr, lg = _disc_out(0)
    loss = L.gan_loss("least_squares", out, mode)
    if mode == "generator_loss":
        want = 0.5 * ((out.D_gen - 1.0) ** 2).mean()
    else:
        want = 0.5 * (((out.D_real - 1.0) ** 2).mean() + (out.D_gen ** 2).mean())
    assert torch.allclose(loss, want, rtol=0, atol=0)
    loss.backward()
    assert lg.grad is not None and (mode == "generator_loss") == (lr.grad is None)


def test_invalid_gan_loss_type_raises_like_the_reference():
    out, _, _ = _disc_out(1)
    with pytest.raises(ValueError):
        L.gan_loss("hinge", out, "generator_loss")


@pytest.mark.parametrize("mode", ["generator_loss", "discriminator_loss"])
def test_least_squares_gan_loss_equals_the_references(mode):
    gold = np.load(GOLDEN)
    out, lr, lg = _disc_out(2)
    ours = L.gan_loss("least_squares", out, mode)
    ours.backward()
    # the gradients are elementwise (bit-exact on any CPU); the loss is a mean whose summation order depends on the CPU
    assert float(ours) == pytest.approx(float(gold[f"ls_gan.{mode}.loss"]), rel=1e-6, abs=0)
    assert torch.equal(lg.grad, torch.from_numpy(gold[f"ls_gan.{mode}.grad_gen"]))
    assert (lr.grad is not None) == bool(gold[f"ls_gan.{mode}.has_grad_real"])
    if lr.grad is not None:
        assert torch.equal(lr.grad, torch.from_numpy(gold[f"ls_gan.{mode}.grad_real"]))
