"""Generate tests/golden/dropin_reference.npz from the REAL reference's callers -- TEST INFRASTRUCTURE, needs a checkout of
the reference (HIFIC_REFERENCE_ROOT, see oracle/ref_shim.py).

    HIFIC_REFERENCE_ROOT=<checkout> python oracle/make_golden_dropin.py

Runs the reference's unmodified `train.train()` (two generator + two discriminator iterations, train.py:89-200) and
`compress.compress_and_decompress()` (compress.py:101-200) on the seeds, images and noise of tests/test_dropin_reference.py
and stores what that test compares the repository's own training loop, checkpoint and compression path against:

  train.*     every value the reference logged (except wall-clock times), the step count, the state_dict key order, the
              direction each parameter moved (a seeded sample of 1.5 M elements; the model has far more) and the
              spectral-norm u / v buffers after training;
  ckpt.*      the layout of `utils.save_model`'s checkpoint: keys, state_dict names / shapes, optimizer state layout;
  compress.*  the metrics table, the .hfc files and the reconstructions compress.py wrote for two 176 x 176 PNGs from a
              checkpoint of the initial weights.

The model's weights are NOT stored: the repository's Model draws the reference's initial weights bit for bit under the
same seed (checked through the stored per-tensor sums of the initial state_dict).
"""
import glob
import logging
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


class _Py2Iter:
    def __init__(self, it):
        self._it = it

    def __iter__(self):
        return self

    def __next__(self):
        return next(self._it)

    next = __next__                      # train.py:160 `test_loader_iter.next()` (py2 bit rot, SURVEY.md section 8c)


class _Loader:
    """The loaders' interface: batches of (data, bpp)."""

    def __init__(self, batches):
        self.batches = batches

    def __iter__(self):
        return _Py2Iter(iter(self.batches))

    def __len__(self):
        return len(self.batches)


def _optimizers(model, args):
    """train.py:287-300."""
    import itertools
    amort = itertools.chain.from_iterable([am.parameters() for am in model.amortization_models])
    return dict(amort=torch.optim.Adam(amort, lr=args.learning_rate),
                hyper=torch.optim.Adam(model.Hyperprior.hyperlatent_likelihood.parameters(), lr=args.learning_rate),
                disc=torch.optim.Adam(model.Discriminator.parameters(), lr=args.learning_rate))


def delta_sample(T, sd, init):
    """(moved, positive) bits of `sd - init` at the test's seeded positions of the concatenated trainable tensors."""
    d = T._trainable_delta(sd, init)
    d = d.numpy()[T._sample_index(d.numel())]
    return np.packbits(d != 0), np.packbits(d > 0)


def main():
    import tempfile
    from collections import defaultdict

    import pandas as pd
    import test_dropin_reference as T
    from oracle import ref_shim
    assert ref_shim.available(), "set HIFIC_REFERENCE_ROOT to a checkout of the reference"
    tmp = tempfile.mkdtemp(prefix="hfc_golden_dropin_")
    torch.set_num_threads(os.cpu_count())
    ref_shim.install_ans()
    import compress as ref_compress
    import default_config as dc
    import src.model as ref_model
    import train as ref_train
    from src.helpers import utils as ref_utils

    args = T._args(dc, tmp, "ref")
    logger = logging.getLogger("ref")
    torch.manual_seed(7)
    storage, storage_test = defaultdict(list), defaultdict(list)
    model = ref_model.Model(args, logger, storage, storage_test, model_type=args.model_type)
    with T._FixedNoise():
        model, ckpt = ref_train.train(args, model, _Loader(T._batches(4, 1)), _Loader(T._batches(2, 2)),
                                      torch.device("cpu"), logger, _optimizers(model, args))
    out = {"train.step_counter": np.array(model.step_counter)}
    for tag, st in (("storage", storage), ("storage_test", storage_test)):
        keys = sorted(k for k in st if k != "time")
        out[f"train.{tag}.keys"] = np.array(keys)
        for k in keys:
            out[f"train.{tag}.{k}"] = np.asarray(st[k], dtype=np.float64)
    sd = model.state_dict()
    out["train.state_keys"] = np.array(list(sd))
    torch.manual_seed(7)
    init_args = T._args(dc, tmp, "init")
    init_model = ref_model.Model(init_args, logging.getLogger("init"), model_type=dc.ModelTypes.COMPRESSION_GAN)
    init = init_model.state_dict()
    out["train.init_sums"] = np.array([float(v.double().sum()) for v in init.values()])
    out["train.moved"], out["train.positive"] = delta_sample(T, sd, init)
    uv = [k for k in sd if "weight_u" in k or "weight_v" in k]
    out["train.uv_keys"] = np.array(uv)
    for k in uv:
        out[f"train.uv.{k}"] = sd[k].numpy()

    ck = torch.load(ckpt, weights_only=False)
    out["ckpt.keys"] = np.array(sorted(ck))
    for part in ("model_state_dict", "discriminator_state_dict"):
        out[f"ckpt.{part}.names"] = np.array(list(ck[part]))
        out[f"ckpt.{part}.shapes"] = np.array([",".join(map(str, v.shape)) for v in ck[part].values()])
    for part in ("compression_optimizer_state_dict", "hyperprior_optimizer_state_dict", "discriminator_optimizer_state_dict"):
        o = ck[part]
        out[f"ckpt.{part}.n_params"] = np.array([len(g["params"]) for g in o["param_groups"]])
        out[f"ckpt.{part}.state_shapes"] = np.array([f"{i}:{k}:" + ",".join(map(str, v.shape)) for i, s in o["state"].items()
                                                     for k, v in sorted(s.items()) if torch.is_tensor(v)])
    out["ckpt.steps"] = np.array(ck["steps"])

    # compress.py on two PNGs from a checkpoint of the initial weights (which the test's Model reproduces exactly)
    ckpt = ref_utils.save_model(init_model, _optimizers(init_model, init_args), np.nan, 0, torch.device("cpu"),
                                args=init_args, logger=logging.getLogger("init"))
    img_dir, out_dir = T._write_eval_images(tmp), os.path.join(tmp, "out_ref")
    tables = {}
    pd.DataFrame.to_hdf = lambda self, path, **kw: tables.__setitem__(path, self.copy())   # PyTables is not installed
    base = {k: getattr(dc.args, k) for k in dir(dc.args) if not k.startswith("_")}
    base.update(ckpt_path=ckpt, image_dir=img_dir, output_dir=out_dir, batch_size=1, reconstruct=False, save=True,
                metrics=True, normalize_input_image=False)
    ref_compress.compress_and_decompress(ref_utils.Struct(**base))
    (_, df), = tables.items()
    df = df.sort_values("input_filename")          # the loader lists the folder in file-system order
    out["compress.columns"] = np.array(list(df.columns))
    for col in ("q_bpp", "LPIPS", "PSNR", "MS_SSIM"):
        out[f"compress.{col}"] = df[col].to_numpy(dtype=np.float64)
    from PIL import Image
    for i, f in enumerate(sorted(glob.glob(os.path.join(out_dir, "*.hfc")))):
        out[f"compress.hfc{i}"] = np.frombuffer(open(f, "rb").read(), dtype=np.uint8)
    for i, f in enumerate(sorted(glob.glob(os.path.join(out_dir, "*_RECON*.png")))):
        out[f"compress.recon{i}"] = np.asarray(Image.open(f).convert("RGB"))
    path = os.path.join(ROOT, "tests", "golden", "dropin_reference.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
