"""CPU: the `-LMM` variant (HyperpriorDLMM, src/hyperprior.py:340-458).

  * the oracle restatement against tests/golden/dlmm_c8.npz, produced by the REAL reference module under seed 21
    (oracle/make_golden_dlmm.py): forward and gradients bit-exact -- with the weights taken from the PRODUCT's mirror module
    built under the same seed, which also proves the constructor draws its parameters in the reference's order;
  * the closed-form backward the CUDA kernel evaluates (tests/emulation.py: dlmm_likelihood_bwd mirrors csrc/dlmm.cu line
    by line) against torch autograd, both gate directions;
  * the product's host logic (module, inference + training plans, autograd Functions) through emulated entry points
    against the same golden values.  The kernels themselves are checked by tests/test_gpu_zzdlmm.py on a GPU.
"""
import os

import numpy as np
import pytest
import torch

import emulation as E
from hific_b200 import hyperprior
from oracle import hific_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dlmm_c8.npz")
FIELDS = ("decoded", "latent_nbpp", "hyperlatent_nbpp", "total_nbpp", "latent_qbpp", "hyperlatent_qbpp", "total_qbpp")
GRAD_KEYS = ("analysis_net.conv1.weight", "synthesis_DLMM_params.conv_out.weight", "synthesis_DLMM_params.conv3.bias",
             "synthesis_DLMM_params.conv3.weight", "hyperlatent_likelihood.H_1")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


def mirror():
    torch.manual_seed(21)
    return hyperprior.HyperpriorDLMM(bottleneck_capacity=8)


@pytest.fixture
def eight_threads():
    """The stored gradients are reproduced bit for bit with eight or more intra-op threads: the CPU convolution's
    weight-gradient reduction sums in an order that depends on the thread count, and fewer threads give other last bits."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def test_oracle_and_constructor_parity_with_the_reference(gold, eight_threads):
    hp = mirror()
    sd = {"Hyperprior." + k: v.detach() for k, v in hp.state_dict().items()}
    y, nz, ny = (torch.from_numpy(gold[k]) for k in ("y", "noise_z", "noise_y"))
    for training in (True, False):
        tag = "train" if training else "eval"
        sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        yy = y.clone().requires_grad_(True)
        o = O.hyperprior_dlmm_forward(sdg, yy, (256, 256), training, nz, ny)
        for f in FIELDS:
            assert np.array_equal(getattr(o, f).detach().numpy(), gold[f"{tag}.{f}"]), (tag, f)
        if training:
            (o.total_nbpp * 1000.0 + o.decoded.square().mean()).backward()
            assert np.array_equal(yy.grad.numpy(), gold["train.grad.y"])
            for k in GRAD_KEYS:
                assert np.array_equal(sdg["Hyperprior." + k].grad.numpy(), gold["train.grad." + k]), k


@pytest.mark.parametrize("kind", ["gaussian", "logistic"])
@pytest.mark.parametrize("upstream", [-0.37, 0.8])
def test_closed_form_backward_matches_autograd(kind, upstream):
    g = torch.Generator().manual_seed(3)
    n, c, k, h, w = 2, 5, 4, 6, 7
    x = (torch.randn((n, c, h, w), generator=g) * 6).requires_grad_(True)      # far tails: pmf below the 1e-9 bound
    params = torch.randn((n, 3 * c * k, h, w), generator=g)
    params[:, 2 * c * k:] = params[:, 2 * c * k:] * 2 - 2.5                     # log-scales on both sides of -3
    params[:, c * k:2 * c * k] *= 3
    params = params.requires_grad_(True)
    noise = torch.rand((n, c, h, w), generator=g) - 0.5
    dd = torch.randn((n, c, h, w), generator=g)
    L = O.dlmm_log_likelihood(x + noise, params, kind)
    dec = x + (torch.floor(x + 0.5) - x).detach()
    (upstream * L.sum() + (dec * dd).sum()).backward()
    dx, dp = E.dlmm_likelihood_bwd(x.detach(), params.detach(), noise, dd, torch.tensor([upstream]), kind)
    assert ((dx - x.grad).norm() / x.grad.norm()).item() < 1e-5
    assert ((dp - params.grad).norm() / params.grad.norm()).item() < 1e-5
    clamped = (params[:, 2 * c * k:] < -3).float().mean().item()
    assert 0.2 < clamped < 0.8


def test_product_host_logic_matches_the_reference(gold):
    """HyperpriorDLMM of the product under emulated entry points: train-mode forward + backward and eval-mode forward
    against the reference's values.  Tolerances: fp16 activations / bf16 gradient operands of the emulated kernels."""
    y, nz, ny = (torch.from_numpy(gold[k]) for k in ("y", "noise_z", "noise_y"))
    with E.training_cpu_emulation():
        from oracle.ref_shim import NoiseFeeder
        hp = mirror().train()
        yy = y.clone().requires_grad_(True)
        with NoiseFeeder([nz, ny]):
            info = hp(yy, spatial_shape=(256, 256))
        (info.total_nbpp * 1000.0 + info.decoded.square().mean()).backward()
        grads = {k: v.grad for k, v in hp.named_parameters()}
        for f in FIELDS[1:]:
            assert abs(float(getattr(info, f)) - float(gold[f"train.{f}"])) < 5e-3 * abs(float(gold[f"train.{f}"])), f
        assert torch.equal(info.decoded.detach(), torch.from_numpy(gold["train.decoded"]))
        rel = lambda a, b: ((a - b).norm() / b.norm()).item()
        assert rel(yy.grad, torch.from_numpy(gold["train.grad.y"])) < 5e-2
        for k in GRAD_KEYS:
            assert rel(grads[k], torch.from_numpy(gold["train.grad." + k])) < 5e-2, k
        hp.eval()
        with torch.no_grad(), NoiseFeeder([nz, ny]):
            info = hp(y, spatial_shape=(256, 256))
        for f in FIELDS[1:]:
            assert abs(float(getattr(info, f)) - float(gold[f"eval.{f}"])) < 5e-3 * abs(float(gold[f"eval.{f}"])), f
        assert torch.equal(info.decoded, torch.from_numpy(gold["eval.decoded"]))
        params = hp.synthesis_DLMM_params(torch.floor(hp.analysis_net(y) + 0.5))
        want = torch.from_numpy(gold["eval.dlmm_params"])
        assert rel(params, want) < 3e-3


@pytest.fixture(scope="module")
def host_kernels(tmp_path_factory):
    """The per-element code of csrc/dlmm.cu (csrc/dlmm_math.cuh) compiled for the HOST with g++."""
    import ctypes
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    so = str(tmp_path_factory.mktemp("dlmm") / "dlmm_math_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-x", "c++",
                    os.path.join(here, "dlmm_math_host.cpp"), "-o", so], check=True)
    return ctypes.CDLL(so)


@pytest.mark.parametrize("kind", ["gaussian", "logistic"])
@pytest.mark.parametrize("shape", [(2, 5, 4, 6, 7), (1, 8, 2, 1, 3), (3, 16, 8, 4, 4)])
def test_kernel_element_code_on_the_host(host_kernels, kind, shape):
    """The functions every CUDA thread runs, executed on the CPU: forward sums / decoded against the oracle, gradients
    against torch autograd (through the closed-form stand-in, itself checked above) -- float32 libm vs torch: 1e-5."""
    import ctypes
    n, c, k, h, w = shape
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn((n, c, h, w), generator=g) * 5
    params = torch.randn((n, 3 * c * k, h, w), generator=g)
    params[:, 2 * c * k:] = params[:, 2 * c * k:] * 2 - 2.5
    params[:, c * k:2 * c * k] *= 3
    noise = torch.rand((n, c, h, w), generator=g) - 0.5
    dd = torch.randn((n, c, h, w), generator=g)
    lt = {"gaussian": 0, "logistic": 1}[kind]
    fp = lambda t: ctypes.c_void_p(t.data_ptr())
    for st in (1, 0):
        dec = torch.empty_like(x)
        sums = torch.zeros(2, dtype=torch.float64)
        host_kernels.dlmm_forward_host(fp(x), fp(noise), fp(params), n, c, k, h * w, lt, st, fp(dec), fp(sums))
        want_dec, want = E.dlmm_likelihood(x, params, noise, kind, bool(st))
        assert torch.equal(dec, want_dec)
        assert torch.allclose(sums, want, rtol=1e-5)
    for upstream in (-0.37, 0.8):
        dx, dp = torch.empty_like(x), torch.empty_like(params)
        host_kernels.dlmm_backward_host(fp(x), fp(noise), fp(params), fp(dd), ctypes.c_float(upstream), n, c, k, h * w, lt,
                                        fp(dx), fp(dp))
        want_dx, want_dp = E.dlmm_likelihood_bwd(x, params, noise, dd, torch.tensor([upstream]), kind)
        assert ((dx - want_dx).norm() / want_dx.norm()).item() < 1e-5
        assert ((dp - want_dp).norm() / want_dp.norm()).item() < 1e-5


def test_model_level_lmm_uses_the_dlmm_channel_count():
    """`Model(use_latent_mixture_model=True)` (`train.py -LMM`): the reference overrides `args.latent_channels` with
    `args.latent_channels_DLMM` before building ANY sub-network (src/model.py:53-54); without the override the shipped
    config (220 channels) trips `HyperpriorDLMM`'s `bottleneck_capacity <= 128` assertion (ADVICE r1).  Construct, run a
    training-mode forward + backward and an eval forward through the emulated entry points."""
    import logging
    from hific_b200.config import mse_lpips_args
    from hific_b200.model import Model
    cfg = mse_lpips_args()
    cfg.use_latent_mixture_model, cfg.latent_channels_DLMM, cfg.n_residual_blocks = True, 8, 1
    cfg.image_dims, cfg.latent_dims, cfg.batch_size = (3, 128, 128), (8, 8, 8), 1
    torch.manual_seed(0)
    m = Model(cfg, logging.getLogger("lmm"))
    assert m.args.latent_channels == 8
    assert m.Encoder.conv_block_out[1].weight.shape[0] == 8 and m.Generator.conv_block_init[2].weight.shape[1] == 8
    assert type(m.Hyperprior).__name__ == "HyperpriorDLMM" and m.Hyperprior.bottleneck_capacity == 8
    x = torch.rand((1, 3, 128, 128))
    with E.train_step_cpu_emulation():
        m.train()
        inter, info = m.compression_forward(x)
        assert inter.reconstruction.shape == x.shape and torch.isfinite(inter.n_bpp) and torch.isfinite(inter.q_bpp)
        (inter.n_bpp + m.distortion_loss(inter.reconstruction, inter.input_image) * 1e-3).backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.Encoder.parameters())
        assert all(p.grad is not None for p in m.Hyperprior.synthesis_DLMM_params.parameters())
        m.eval()
        with torch.no_grad():
            inter2, _ = m.compression_forward(x)
        assert inter2.reconstruction.shape == x.shape and float(inter2.q_bpp) > 0
