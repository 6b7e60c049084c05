"""CPU: the host glue of `Model.compress` / `Model.decompress` (hific_b200.model / hyperprior / compression.*) and the C
host coder, end to end against the messages the REAL reference's `Model.compress` produced for the same weights and
images (tests/golden/entropy_coding.npz, model_m1 = batch 1 ragged 100x144, model_m2 = batch 2).  The CUDA entry points
are swapped for the oracle's CPU arithmetic (tests/emulation.py) -- with bit-identical latents the messages, the
shapes, the Shannon estimates and the reconstruction must be the reference's."""
import logging
import os

import numpy as np
import pytest
import torch

from hific_b200 import synth
from hific_b200.compression import compression_utils
from hific_b200.config import ModelModes, mse_lpips_args
from hific_b200.model import Model
from emulation import cpu_emulation

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "entropy_coding.npz")


@pytest.fixture(scope="module")
def model():
    m = Model(mse_lpips_args(), logging.getLogger("glue"), model_mode=ModelModes.EVALUATION)
    res = m.load_state_dict(synth.synth_state_dict(0), strict=False)
    assert not res.unexpected_keys
    m.eval()
    m.Hyperprior.hyperprior_entropy_model.build_tables()          # compress.py:61,122
    return m


@pytest.fixture
def one_thread():
    """The stored reconstructions were decoded with one intra-op thread.  The fp32 convolutions of the emulated generator
    sum in an order that depends on the thread count (up to 2e-6 apart at 4 or more threads), so decode with one too."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name,b,h,w", [("m1", 1, 100, 144), ("m2", 2, 96, 128)])
def test_model_compress_decompress_reproduces_the_reference(model, name, b, h, w, tmp_path, one_thread):
    g = np.load(GOLDEN)
    x = synth.synth_image(b, h, w, 30 + b)
    with cpu_emulation():
        co = model.compress(x, silent=True)
        assert np.array_equal(co.hyperlatents_encoded, g[f"model_{name}.hyperlatents_encoded"])
        assert np.array_equal(co.latents_encoded, g[f"model_{name}.latents_encoded"])
        shapes = (list(co.hyperlatent_spatial_shape) + list(co.spatial_shape) + list(co.hyper_coding_shape)
                  + list(co.latent_coding_shape) + [co.batch_shape])
        assert shapes == list(g[f"model_{name}.shapes"])
        got = np.array([co.hyperlatent_bpp, co.latent_bpp, co.total_bpp, co.hyperlatent_bits, co.latent_bits, co.total_bits])
        np.testing.assert_allclose(got, g[f"model_{name}.bpp"], rtol=1e-6)
        # through the .hfc container and back, then decode
        p = str(tmp_path / f"{name}.hfc")
        actual_bpp, theoretical_bpp = compression_utils.save_compressed_format(co, p)
        assert abs(theoretical_bpp - co.total_bpp) < 1e-9 and actual_bpp > 0
        rec = model.decompress(compression_utils.load_compressed_format(p))
    assert tuple(rec.shape) == (b, 3, h, w)
    np.testing.assert_allclose(rec.numpy(), g[f"model_{name}.reconstruction"], rtol=0, atol=1e-6)


def test_compress_requires_evaluation_mode():
    m = Model(mse_lpips_args(), logging.getLogger("glue"))
    with pytest.raises(AssertionError):
        m.compress(torch.zeros(1, 3, 96, 96))
    assert not hasattr(m.Hyperprior, "prior_entropy_model")       # tables only in EVALUATION mode (model.py:64-66)
