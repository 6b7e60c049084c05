"""The drop-in claim (north_star: "train.py and compress.py drop in unchanged"; VERDICT r1 row g), against stored outputs of
the reference (tests/golden/dropin_reference.npz, written by oracle/make_golden_dropin.py).

The golden file holds what the reference's UNMODIFIED callers produced -- `train.py`'s `train()` (the alternating G / D
loop, `test()`, `utils.log`, `utils.save_model`) and `compress.py`'s `compress_and_decompress()` (`utils.load_model`,
`build_tables`, `Model.compress` / `Model.decompress`, the `.hfc` container, metrics) -- on the seeds, images and noise
below.  The tests run the same sequence of calls on the `hific_b200` mirrors (`Model`, the loop helpers of
`hific_b200.train_ddp`, `compression_utils`) and compare the logged losses / rates, the direction every parameter moved,
the spectral-norm buffers, the checkpoint layout, the metrics table and the compressed files.  There is no GPU here, so
the mirror's CUDA entry points are replaced by tests/emulation.py's CPU stand-ins (fp16-operand arithmetic of the
kernels); what these tests pin is the HOST contract, while the kernels themselves are pinned by the `-m gpu` tests.
The `sample_noise` Generator test compares with tests/golden/noise_generator_ls_gan.npz (oracle/make_golden_noise_gan.py).
"""
import logging
import os
from collections import defaultdict
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import emulation as E
import hific_b200  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "noise_generator_ls_gan.npz")
GOLDEN_DROPIN = os.path.join(HERE, "golden", "dropin_reference.npz")

IMG = 128          # smallest size the hyper-analysis reflect padding accepts (latents 8 x 8, hyper-latents 2 x 2)
N_RES = 2          # residual blocks (keeps the CPU runs short; the class code is the same for 9)
EV = 176           # compress.py images: MS-SSIM needs > 160 pixels; 176 / 16 = 11 latent rows -> pad-to-4 of the latents
N_SAMPLE = 1_500_000   # parameter elements whose direction of travel is stored (seeded positions)


# ----------------------------------------------------------------------------------------------------------------------
# inputs shared with oracle/make_golden_dropin.py
# ----------------------------------------------------------------------------------------------------------------------
def _batches(n, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand((2, 3, IMG, IMG), generator=g), torch.full((2,), 8.0)) for _ in range(n)]


def _args(dc, tmp, name):
    """train.py's arguments for a two-iteration COMPRESSION_GAN run; `dc` is the reference's `default_config` or
    `hific_b200.config` (same names and values)."""
    base = {k: getattr(dc.hific_args, k) for k in dir(dc.hific_args) if not k.startswith("_")}   # incl. inherited
    d = os.path.join(str(tmp), name)
    base.update(dict(
        name=name, model_type=dc.ModelTypes.COMPRESSION_GAN, model_mode=dc.ModelModes.TRAINING, regime="low",
        image_dims=(3, IMG, IMG), batch_size=2, latent_dims=(220, IMG // 16, IMG // 16), n_residual_blocks=N_RES,
        n_epochs=1, n_steps=100, log_interval=100, save_interval=10_000, discriminator_steps=1, gpu=0, multigpu=False,
        normalize_input_image=False, use_latent_mixture_model=False, sample_noise=False, noise_dim=0,
        ignore_schedule=True, lr_schedule=dict(vals=[1., 0.1], steps=[500000]), learning_rate=1e-4,
        target_rate=0.14, lambda_A=2 ** 1, lambda_B=2 ** (-4), weight_decay=1e-6,
        tensorboard_runs=os.path.join(d, "tb"), storage_save=os.path.join(d, "storage"),
        figures_save=os.path.join(d, "figures"), checkpoints_save=os.path.join(d, "checkpoints"), snapshot=d))
    for sub in ("tb", "storage", "figures", "checkpoints"):
        os.makedirs(os.path.join(d, sub), exist_ok=True)
    return SimpleNamespace(**base)


class _FixedNoise:
    """Both runs consume the same quantisation noise: the k-th uniform_(-0.5, 0.5) draw of a given shape is seeded by
    (k, shape), whoever asks for it."""

    def __enter__(self):
        self._orig, self.calls = torch.nn.init.uniform_, 0
        outer = self

        def fake(t, a=0.0, b=1.0):
            if (a, b) != (-0.5, 0.5):
                return outer._orig(t, a, b)
            g = torch.Generator().manual_seed(1000 + outer.calls)
            outer.calls += 1
            with torch.no_grad():
                t.copy_(torch.rand(t.shape, generator=g) - 0.5)
            return t
        torch.nn.init.uniform_ = fake
        return self

    def __exit__(self, *e):
        torch.nn.init.uniform_ = self._orig


def _write_eval_images(tmp):
    """Two EV x EV PNGs (smooth patterns + noise) for compress.py; returns their directory."""
    from PIL import Image
    img_dir = os.path.join(str(tmp), "images")
    os.makedirs(img_dir, exist_ok=True)
    g = np.random.default_rng(5)
    for i in range(2):
        yy, xx = np.mgrid[0:EV, 0:EV]
        img = np.stack([127 + 100 * np.sin(xx / (7.0 + i) + c) * np.cos(yy / (11.0 + c)) for c in range(3)], -1)
        img = np.clip(img + g.normal(0, 6, img.shape), 0, 255).astype(np.uint8)
        Image.fromarray(img).save(os.path.join(img_dir, f"img{i}.png"))
    return img_dir


def _sample_index(n):
    return np.sort(np.random.default_rng(0).choice(n, N_SAMPLE, replace=False))


def _trainable_delta(sd, init):
    return torch.cat([(sd[k] - init[k]).flatten() for k in sd if sd[k].is_floating_point()
                      and "weight_u" not in k and "weight_v" not in k])


# ----------------------------------------------------------------------------------------------------------------------
# the reference's callers, restated on the mirrors
# ----------------------------------------------------------------------------------------------------------------------
def _new_model(args, storage=None, storage_test=None, mode="training"):
    from hific_b200.model import Model
    torch.manual_seed(7)
    return Model(args, logging.getLogger(args.name), storage if storage is not None else defaultdict(list),
                 storage_test if storage_test is not None else defaultdict(list), model_mode=mode,
                 model_type=args.model_type)


def _sqdiff_sum(a, b, scale=255.0):
    return (((a - b) * scale).double() ** 2).sum().reshape(1)


def _gan_sums(logits):
    real, gen = logits.double().chunk(2)
    F = torch.nn.functional
    return torch.stack([F.softplus(-real).sum(), F.softplus(gen).sum(), F.softplus(-gen).sum(),
                        torch.sigmoid(real).sum(), torch.sigmoid(gen).sum()])


def _train(args):
    """train.py:89-200 with one epoch over 4 batches: generator / discriminator iterations alternate, and after the first
    generator iteration (step_counter % log_interval == 1) `test()` runs the train batch and a test batch in eval mode
    and `utils.log` records the epoch and the running mean loss."""
    from hific_b200 import ops, train_ddp
    storage, storage_test = defaultdict(list), defaultdict(list)
    model = _new_model(args, storage, storage_test)
    opts = train_ddp.make_optimizers(model, args, adam=lambda params, lr: torch.optim.Adam(params, lr=lr))
    model.perceptual_loss                # built before the noise feeder, as the reference builds it in Model.__init__
    test_batches = iter(_batches(2, 2))
    train_generator, d_steps, epoch_loss, epoch_test_loss = True, 0, [], []
    model.train()
    with E.gan_model_cpu_emulation(), _FixedNoise():
        for data, _ in _batches(4, 1):
            losses = model(data, train_generator=train_generator)
            if train_generator:
                train_ddp.optimize_compression_loss(model, losses["compression"], opts["amort"], opts["hyper"], None, None)
                train_generator = False
            else:
                train_ddp.optimize_loss(losses["disc"], opts["disc"], None, None, 1)
                d_steps += 1
                if d_steps == args.discriminator_steps:
                    d_steps, train_generator = 0, True
                continue
            if model.step_counter % args.log_interval == 1:
                epoch_loss.append(losses["compression"].item())
                storage["epoch"].append(0)
                storage["mean_compression_loss"].append(float(np.mean(epoch_loss)))
                model.eval()             # the no-grad loss reductions, in torch
                with torch.no_grad(), pytest.MonkeyPatch.context() as mp:
                    mp.setattr(ops, "sqdiff_sum", _sqdiff_sum)
                    mp.setattr(ops, "gan_sums", _gan_sums)
                    model(data, return_intermediates=True, writeout=False)
                    test_losses, _ = model(next(test_batches)[0], return_intermediates=True, writeout=True)
                epoch_test_loss.append(test_losses["compression"].item())
                storage_test["epoch"].append(0)
                storage_test["mean_compression_loss"].append(float(np.mean(epoch_test_loss)))
                model.train()
                for opt in opts.values():
                    train_ddp.update_lr(args, opt, model.step_counter, model.logger)
    ckpt = train_ddp.save_model(model, opts, 0, args, model.logger)
    return model, ckpt, storage, storage_test


def _ms_ssim(x, y, data_range=255.0):
    """Multi-scale SSIM (Wang, Simoncelli & Bovik 2003) as compress.py reports it: 11-tap Gaussian window (sigma 1.5)
    without padding, K = (0.01, 0.03), five scales with the standard weights, 2 x 2 average pooling between scales, negative
    contrast-structure terms clamped to zero; mean over images and channels."""
    import torch.nn.functional as F
    c = x.shape[1]
    t = torch.arange(11, dtype=x.dtype) - 5
    w = torch.exp(-t ** 2 / (2 * 1.5 ** 2))
    w = (w / w.sum()).reshape(1, 1, 1, 11).repeat(c, 1, 1, 1)

    def blur(a):
        return F.conv2d(F.conv2d(a, w, groups=c), w.transpose(2, 3), groups=c)

    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    weights = torch.tensor([0.0448, 0.2856, 0.3001, 0.2363, 0.1333], dtype=x.dtype)
    terms = []
    for level in range(5):
        mx, my = blur(x), blur(y)
        sxx, syy, sxy = blur(x * x) - mx * mx, blur(y * y) - my * my, blur(x * y) - mx * my
        cs = ((2 * sxy + c2) / (sxx + syy + c2))
        if level < 4:
            terms.append(torch.relu(cs.flatten(2).mean(-1)))
            pad = [s % 2 for s in x.shape[2:]]
            x, y = F.avg_pool2d(x, 2, padding=pad), F.avg_pool2d(y, 2, padding=pad)
        else:
            ssim = ((2 * mx * my + c1) / (mx * mx + my * my + c1)) * cs
            terms.append(torch.relu(ssim.flatten(2).mean(-1)))
    return torch.prod(torch.stack(terms) ** weights.view(-1, 1, 1), dim=0).mean(1)


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN_DROPIN)


@pytest.fixture(scope="module")
def run(tmp_path_factory):
    from hific_b200 import config
    tmp = tmp_path_factory.mktemp("dropin")
    torch.set_num_threads(os.cpu_count())
    args = _args(config, tmp, "dropin")
    model, ckpt, storage, storage_test = _train(args)
    return dict(tmp=tmp, args=args, model=model, ckpt=ckpt, storage=storage, storage_test=storage_test)


def test_train_py_runs_unchanged_on_the_mirror(run, gold):
    """Two generator + two discriminator iterations of train.py's loop: same step count, same logged keys, losses and rates
    within the fp16-operand tolerance, and the parameters moved the way the reference's did."""
    model, storage, storage_test = run["model"], run["storage"], run["storage_test"]
    assert model.step_counter == int(gold["train.step_counter"]) == 2       # counts generator iterations (src/model.py:352)
    assert type(model.Encoder).__module__ == "hific_b200.network.encoder"
    assert type(model.Discriminator).__module__ == "hific_b200.network.discriminator"
    assert run["ckpt"] and os.path.exists(run["ckpt"])
    for tag, store in (("storage", storage), ("storage_test", storage_test)):
        assert sorted(store) == list(gold[f"train.{tag}.keys"]), tag          # wall-clock `time` is not stored
        assert len(store) >= 10
        for k in store:
            a, b = gold[f"train.{tag}.{k}"], np.asarray(store[k], dtype=np.float64)
            assert a.shape == b.shape, k
            assert np.allclose(a, b, rtol=3e-2, atol=3e-3), (k, a, b)
    sd = model.state_dict()
    assert list(sd) == list(gold["train.state_keys"])
    init = _new_model(run["args"]).state_dict()
    # the mirror draws the reference's initial weights: float64 sums equal up to the CPU's summation order
    sums = np.array([float(v.double().sum()) for v in init.values()])
    assert np.allclose(sums, gold["train.init_sums"], rtol=1e-9, atol=1e-9)
    # after 2 Adam steps per group the parameters of both runs left the common initialisation in the same direction
    d = _trainable_delta(sd, init)
    d = d.numpy()[_sample_index(d.numel())]
    n = len(d)
    ref_moved = np.unpackbits(gold["train.moved"])[:n].astype(bool)
    ref_pos = np.unpackbits(gold["train.positive"])[:n].astype(bool)
    agree = int(np.sum(ref_moved & (d != 0) & ((d > 0) == ref_pos)))
    total = int(ref_moved.sum())
    assert total > 1_000_000 and agree / total > 0.97, (agree, total)
    assert list(gold["train.uv_keys"]) == [k for k in sd if "weight_u" in k or "weight_v" in k]
    for k in gold["train.uv_keys"]:                        # spectral-norm buffers: updated in place by both
        assert torch.allclose(torch.from_numpy(gold[f"train.uv.{k}"]), sd[k], atol=2e-3), k
        assert not torch.equal(sd[k], init[k]), k


def test_checkpoints_are_interchangeable(run, gold):
    """The checkpoint has utils.save_model's layout (same keys, state_dict names / shapes, optimizer state layout as the
    reference's), so either implementation's `utils.load_model` reads the other's; and it round trips into the mirror."""
    ck = torch.load(run["ckpt"], weights_only=False)
    assert sorted(ck) == list(gold["ckpt.keys"])
    assert ck["steps"] == int(gold["ckpt.steps"])
    for part in ("model_state_dict", "discriminator_state_dict"):
        assert list(ck[part]) == list(gold[f"ckpt.{part}.names"]), part
        assert [",".join(map(str, v.shape)) for v in ck[part].values()] == list(gold[f"ckpt.{part}.shapes"]), part
    for part in ("compression_optimizer_state_dict", "hyperprior_optimizer_state_dict", "discriminator_optimizer_state_dict"):
        o = ck[part]
        assert [len(g["params"]) for g in o["param_groups"]] == list(gold[f"ckpt.{part}.n_params"]), part
        assert [f"{i}:{k}:" + ",".join(map(str, v.shape)) for i, s in o["state"].items() for k, v in sorted(s.items())
                if torch.is_tensor(v)] == list(gold[f"ckpt.{part}.state_shapes"]), part
    m = _new_model(run["args"])
    m.load_state_dict(ck["model_state_dict"], strict=True)
    m.Discriminator.load_state_dict(ck["discriminator_state_dict"], strict=True)
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), run["model"].state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2), k1


def test_compress_py_runs_unchanged_on_the_mirror(run, gold):
    """compress.py's path on two PNG files from the same checkpoint (the initial weights, which both implementations draw
    under seed 7): entropy-coded .hfc files, decoded reconstructions and the metrics table against the reference's; the
    mirror decodes the reference's .hfc files to the reference's reconstructions, and writes the reference's layout."""
    import torchvision
    from PIL import Image
    from hific_b200.compression import compression_utils
    from hific_b200.loss.perceptual import PerceptualLoss
    tmp = run["tmp"]
    img_dir = _write_eval_images(tmp)
    args = SimpleNamespace(**{**vars(run["args"]), "name": "eval"})
    model = _new_model(args, mode="evaluation")
    model.load_state_dict(_new_model(run["args"]).state_dict(), strict=False)   # utils.load_model(..., strict=False)
    model.eval()
    model.Hyperprior.hyperprior_entropy_model.build_tables()           # compress.py:122
    lpips = PerceptualLoss()
    cols = {c: [] for c in ("q_bpp", "LPIPS", "PSNR", "MS_SSIM")}

    def read(path):
        return np.asarray(Image.open(path).convert("RGB"), dtype=np.float64)

    with torch.no_grad(), E.cpu_emulation():
        for i in range(2):
            data = torch.from_numpy(read(os.path.join(img_dir, f"img{i}.png")) / 255.0).permute(2, 0, 1)[None].float()
            co = model.compress(data)
            path = os.path.join(str(tmp), f"img{i}_compressed.hfc")
            compression_utils.save_compressed_format(co, path)
            rec = model.decompress(co)
            cols["q_bpp"].append(float(co.total_bpp))
            cols["LPIPS"].append(float(E.perceptual_forward(lpips, rec, data, normalize=True)))
            r, x = rec.numpy().astype(np.float64) * 255.0, data.numpy().astype(np.float64) * 255.0
            cols["PSNR"].append(float(20 * np.log10(255.0) - 10 * np.log10(np.mean((r - x) ** 2))))
            cols["MS_SSIM"].append(float(_ms_ssim(rec * 255.0, data * 255.0)))
            ref_file = gold[f"compress.hfc{i}"]
            size = os.path.getsize(path)                   # sizes differ only by rounding flips
            assert abs(size - ref_file.size) <= 0.03 * ref_file.size + 16, (i, size, ref_file.size)
            ref_path = os.path.join(str(tmp), f"ref_img{i}_compressed.hfc")
            ref_file.tofile(ref_path)
            ours, theirs = compression_utils.load_compressed_format(path), compression_utils.load_compressed_format(ref_path)
            for f in ("hyperlatent_spatial_shape", "spatial_shape", "hyper_coding_shape", "latent_coding_shape",
                      "batch_shape"):                     # same container layout
                assert tuple(np.atleast_1d(getattr(ours, f))) == tuple(np.atleast_1d(getattr(theirs, f))), f
            # the reference's file decoded by the mirror gives the reference's reconstruction (compress.py:94 writes it)
            out = os.path.join(str(tmp), f"cross_img{i}.png")
            torchvision.utils.save_image(model.decompress(theirs), out, normalize=True)
            a, b = read(out), gold[f"compress.recon{i}"].astype(np.float64)
            psnr = 10 * np.log10(255.0 ** 2 / max(np.mean((a - b) ** 2), 1e-12))
            assert psnr > 40.0, (i, psnr)                  # same symbols; generator arithmetic differs (fp16 operands)
    assert set(cols) <= set(gold["compress.columns"])
    for col, got in cols.items():
        want = gold[f"compress.{col}"]
        assert np.allclose(want, got, rtol=3e-2, atol=1e-3), (col, want, got)


def test_sample_noise_generator_against_the_real_reference():
    """`sample_noise=True` (src/network/generator.py:105-107, 149-161): the real reference Generator's output (stored), the
    oracle's restatement and the mirror (kernel emulation: fp16 operands) on the same weights and the same noise draw;
    identical state_dict keys / shapes.  The mirror draws the reference's weights under the same seed (checked through the
    stored per-tensor sums), so the weights themselves are not stored."""
    from hific_b200.network import generator as mirror_generator
    from oracle import hific_oracle as O
    gold = np.load(GOLDEN)
    torch.manual_seed(9)
    mir = mirror_generator.Generator((220, 8, 8), 2, C=220, n_residual_blocks=2, sample_noise=True, noise_dim=32)
    sd_mir = mir.state_dict()
    assert list(sd_mir) == list(gold["noise_generator.keys"])
    assert [",".join(map(str, v.shape)) for v in sd_mir.values()] == list(gold["noise_generator.shapes"])
    sums = np.array([float(v.double().sum()) for v in sd_mir.values()])
    # same draws: the float64 sums agree up to the summation order, which depends on the CPU and the thread count
    assert np.allclose(sums, gold["noise_generator.sums"], rtol=1e-9, atol=1e-9)
    g = torch.Generator().manual_seed(10)
    y_hat = torch.round(torch.randn((2, 220, 8, 8), generator=g) * 2)
    z = torch.randn((2, 32, 8, 8), generator=g)
    want = torch.from_numpy(gold["noise_generator.output"])
    orig = torch.randn
    torch.randn = lambda *a, **k: z.clone()
    try:
        with torch.no_grad(), E.plan_cpu_emulation():
            got = mir.eval()(y_hat)
    finally:
        torch.randn = orig
    sd = {"Generator." + k: v for k, v in sd_mir.items()}
    with torch.no_grad():
        orc = O.generator_forward(sd, y_hat, n_residual_blocks=2, noise=z)
    # the oracle's noise variant is the reference's arithmetic: equal up to the fp32 summation order of the CPU's convolutions
    assert float((orc - want).norm() / want.norm()) < 1e-6
    assert float((got - want).norm() / want.norm()) < 1e-3
