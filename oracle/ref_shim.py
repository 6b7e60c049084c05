"""Import the UNMODIFIED reference (read-only, a checkout named by HIFIC_REFERENCE_ROOT) -- TEST INFRASTRUCTURE.

Only usable where such a checkout exists; nothing that runs on a GPU machine may depend on it.  Three workarounds, none
touching hot-path arithmetic (SURVEY.md section 8c):
  1. `autograd` (HIPS) is not installed: stubbed (only the host ANS coder uses it);
  2. `skimage` is not installed: stubbed (imported by LPIPS / datasets, unused on the path);
  3. no network: torchvision's `alexnet(pretrained=True)` becomes a seeded random trunk.
"""
import os
import sys
import types

REF_ROOT = os.environ.get("HIFIC_REFERENCE_ROOT", "")


def available():
    return bool(REF_ROOT) and os.path.isdir(os.path.join(REF_ROOT, "src"))


def install():
    if not available():
        raise RuntimeError(f"reference not found at HIFIC_REFERENCE_ROOT={REF_ROOT!r}")
    import numpy as np
    if "autograd" not in sys.modules:
        ag = types.ModuleType("autograd")
        ag.numpy = np
        ag.make_vjp = lambda *a, **k: None
        ext = types.ModuleType("autograd.extend")
        ext.primitive = lambda f: f
        ext.defvjp = lambda *a, **k: None
        ext.vspace = lambda *a, **k: None
        ext.VSpace = object
        ag.extend = ext
        sys.modules["autograd"] = ag
        sys.modules["autograd.numpy"] = np
        sys.modules["autograd.extend"] = ext
    for name in ("skimage", "skimage.measure", "skimage.color", "skimage.transform", "skimage.io"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.compare_ssim = m.structural_similarity = m.imread = lambda *a, **k: None
            sys.modules[name] = m
    import torch
    import torchvision

    orig_alexnet = torchvision.models.alexnet

    def alexnet_offline(pretrained=False, **kw):
        state = torch.random.get_rng_state()
        torch.manual_seed(1234)
        net = orig_alexnet(weights=None)
        torch.random.set_rng_state(state)
        return net

    torchvision.models.alexnet = alexnet_offline
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)


class NoiseFeeder:
    """Replaces torch.nn.init.uniform_ while active so the reference consumes OUR noise tensors, in order
    (hyper-latents first, then latents -- src/hyperprior.py:65 called from :284 and :305)."""

    def __init__(self, noises):
        self.noises = list(noises)
        self.calls = 0

    def __enter__(self):
        import torch
        self._orig = torch.nn.init.uniform_

        def fake(t, a=0.0, b=1.0):
            n = self.noises[self.calls]
            self.calls += 1
            assert tuple(n.shape) == tuple(t.shape), (n.shape, t.shape)
            with torch.no_grad():
                t.copy_(n)
            return t

        torch.nn.init.uniform_ = fake
        return self

    def __exit__(self, *exc):
        import torch
        torch.nn.init.uniform_ = self._orig


def install_ans():
    """Make the reference's vectorised rANS coder (src/compression/entropy_coding.py, ans.py) runnable here.
    Two workarounds, neither changes its arithmetic:
      4. NumPy 2 removed value-based casting: `((RANS_L >> precision) << 32) * freqs` (ans.py:64) with uint32
         `freqs` raises OverflowError (under NumPy 1.x the product is uint64).  `ans.push` is wrapped so that
         starts / freqs arrive as uint64 -- exactly the dtype NumPy 1.x promoted them to.
      5. `substack` (entropy_coding.py:418-446) updates the masked lanes of the message head through HIPS
         autograd's `make_vjp`; without that package the same update is written as a masked assignment.
    """
    install()
    import numpy as np
    from src.compression import ans as vrans
    from src.compression import entropy_coding
    if getattr(vrans, "_hfc_patched", False):
        return
    orig_push = vrans.push

    def push_u64(x, starts, freqs, precisions):
        return orig_push(x, np.asarray(starts, dtype=np.uint64), np.asarray(freqs, dtype=np.uint64), precisions)

    vrans.push = push_u64

    def substack(codec, view_fun):
        def push(message, start, freq, precision, mask):
            head, tail = message
            subhead, tail = vrans.push((view_fun(head, mask), tail), start, freq, precision)
            head = np.copy(head)
            head[mask] = subhead
            return head, tail

        def pop(message, precision, mask, *args, **kwargs):
            head, tail = message
            cf, pop_fun = vrans.pop((view_fun(head, mask), tail), precision)
            subhead, tail = pop_fun(cf, 1)
            head = np.copy(head)
            head[mask] = subhead
            return (head, tail), cf

        return entropy_coding.Codec(push, pop)

    entropy_coding.substack = substack
    vrans._hfc_patched = True
