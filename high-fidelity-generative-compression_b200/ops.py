"""Host wrappers over the libhfc C ABI: torch tensors own the device memory, raw pointers cross
the boundary, work is enqueued on torch's current CUDA stream.  Nothing here computes on the CPU
or falls back to torch operators.
"""
import ctypes
from dataclasses import dataclass, replace

import torch
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import (ACT_LEAKY02, ACT_NONE, ACT_RELU, OUT_NCHW_F32, OUT_NHWC_F16, OUT_NHWC_F32,
                   PAD_REFLECT, PAD_ZERO, PREC_F16, check, lib)

CN_EPS = 1e-3  # ChannelNorm2D eps (reference: src/normalisation/channel.py:35)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(t.data_ptr())


def round_up(v, m):
    return (v + m - 1) // m * m


@dataclass(frozen=True)
class Geom:
    """NHWC 16-bit activation buffer geometry (``hfc_act_geom``)."""
    n: int
    h: int
    w: int
    c: int
    cpad: int
    pt: int = 0
    pl: int = 0
    pb: int = 0
    pr: int = 0

    def c_struct(self):
        return _lib.ActGeom(self.n, self.h, self.w, self.c, self.cpad, self.pt, self.pl, self.pb, self.pr)

    @property
    def shape(self):
        return (self.n, self.h + self.pt + self.pb, self.w + self.pl + self.pr, self.cpad)

    def alloc(self, device):
        return torch.empty(self.shape, dtype=torch.float16, device=device)

    def interior(self, buf):
        """(n, c, h, w) fp32 view of the logical content of an act buffer (tests / debugging)."""
        x = buf[:, self.pt:self.pt + self.h, self.pl:self.pl + self.w, :self.c]
        return x.permute(0, 3, 1, 2).float()


def device_info():
    sm, ma, mi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    check(lib.hfc_device_info(ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi)), "device_info")
    return sm.value, ma.value, mi.value


def launch_count():
    return int(lib.hfc_launch_count())


def nchw_to_act(x, geom, reflect=False, norm=False, gamma=None, beta=None, out=None):
    """fp32 NCHW tensor -> act buffer (optionally ChannelNorm2D first)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
    assert tuple(x.shape) == (geom.n, geom.c, geom.h, geom.w), (tuple(x.shape), geom)
    if out is None:
        out = geom.alloc(x.device)
    g = geom.c_struct()
    gm = gamma.reshape(-1) if gamma is not None else None
    bt = beta.reshape(-1) if beta is not None else None
    check(lib.hfc_nchw_to_act(_ptr(x), ctypes.byref(g), int(reflect), int(norm), _ptr(gm), _ptr(bt),
                              CN_EPS, _ptr(out), _stream()), "nchw_to_act")
    return out


def channelnorm(x_rows, geom, gamma, beta, act=ACT_NONE, reflect=False, res1=None, res2=None,
                want_f32=False, want_act=True, out_act=None, out_f32=None):
    """Stand-alone ChannelNorm2D over NHWC fp32 rows ``x_rows`` of shape (n*h*w, ld)."""
    assert x_rows.dtype == torch.float32 and x_rows.is_contiguous()
    ld = x_rows.shape[-1]
    if want_act and out_act is None:
        out_act = geom.alloc(x_rows.device)
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty((geom.n * geom.h * geom.w, geom.c), dtype=torch.float32, device=x_rows.device)
    g = geom.c_struct()
    check(lib.hfc_channelnorm(_ptr(x_rows), ld, ctypes.byref(g), int(reflect), _ptr(gamma.reshape(-1)),
                              _ptr(beta.reshape(-1)), CN_EPS, act, _ptr(res1), _ptr(res2),
                              _ptr(out_f32 if want_f32 else None), _ptr(out_act if want_act else None),
                              _stream()), "channelnorm")
    return out_act, out_f32


IN_EPS = 1e-5           # torch.nn.InstanceNorm2d default (src/normalisation/instance.py:12-14 does not override it)
_in_ws_cache = {}


def instancenorm_ws(n, c, device):
    """Scratch of hfc_instancenorm / hfc_instancenorm_bwd (double accumulators + per-(n, c) statistics); one buffer per
    device, grown on demand -- the launches that use it are ordered on the current stream."""
    need = int(lib.hfc_instancenorm_ws_bytes(int(n), int(c)))
    buf = _in_ws_cache.get(device)
    if buf is None or buf.numel() * 8 < need:
        buf = _in_ws_cache[device] = torch.empty((need + 7) // 8, dtype=torch.float64, device=device)
    return buf, buf.numel() * 8


def instancenorm(x_rows, geom, gamma, beta, act=ACT_NONE, reflect=False, res1=None, res2=None,
                 want_f32=False, want_act=True, out_act=None, out_f32=None):
    """InstanceNorm2d(affine) over NHWC fp32 rows (use_channel_norm=False variant; src/normalisation/instance.py:7-15):
    the drop-in of `channelnorm` with per-(image, channel) statistics."""
    assert x_rows.dtype == torch.float32 and x_rows.is_contiguous()
    ld = x_rows.shape[-1]
    if want_act and out_act is None:
        out_act = geom.alloc(x_rows.device)
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty((geom.n * geom.h * geom.w, geom.c), dtype=torch.float32, device=x_rows.device)
    g = geom.c_struct()
    ws, ws_bytes = instancenorm_ws(geom.n, geom.c, x_rows.device)
    check(lib.hfc_instancenorm(_ptr(x_rows), ld, ctypes.byref(g), int(reflect), _ptr(gamma.reshape(-1)),
                               _ptr(beta.reshape(-1)), IN_EPS, act, _ptr(res1), _ptr(res2),
                               _ptr(out_f32 if want_f32 else None), _ptr(out_act if want_act else None),
                               _ptr(ws), ws_bytes, _stream()), "instancenorm")
    return out_act, out_f32


class Conv:
    """One convolution / transposed convolution of the hot path bound to fixed geometry.

    Holds the descriptor, the packed (K-major fp16) weights and re-packs them when the source
    parameter changes (``_version`` / storage pointer), so optimizer steps and ``.to()`` are seen.
    """

    def __init__(self, in_geom, cout, k, stride=1, transposed=False, pad_mode=PAD_ZERO, pad=(0, 0, 0, 0),
                 out_mode=OUT_NHWC_F16, out_geom=None, out_reflect=False, act=ACT_NONE, norm=False,
                 window=False, block_n=0, precision=PREC_F16, cluster=(0, 0), wide=0, pair=0, a_bf16=False, b_bf16=False, dgrad=False):
        kh, kw = (k, k) if isinstance(k, int) else k
        pt, pl, pb, pr = pad
        d = _lib.ConvDesc()
        d.inp = in_geom.c_struct()
        d.kh, d.kw, d.stride, d.transposed = kh, kw, stride, int(transposed)
        d.pad_mode = pad_mode
        d.pad_t, d.pad_l, d.pad_b, d.pad_r = pt, pl, pb, pr
        d.cout, d.window = cout, int(window)
        d.out_mode = out_mode
        d.out_reflect, d.act, d.norm = int(out_reflect), act, int(norm)
        d.eps = CN_EPS
        d.block_n, d.precision = block_n, precision
        d.cluster_m, d.cluster_n = cluster
        d.wide = wide
        d.pair = pair
        d.a_bf16, d.b_bf16, d.dgrad = int(a_bf16), int(b_bf16), int(dgrad)
        # output dims
        if transposed:
            oh = (in_geom.h - 1) * stride - 2 * pt + kh + (stride - 1)
            ow = (in_geom.w - 1) * stride - 2 * pl + kw + (stride - 1)
        else:
            oh = (in_geom.h + pt + pb - kh) // stride + 1
            ow = (in_geom.w + pl + pr - kw) // stride + 1
        if out_geom is None:
            out_geom = Geom(in_geom.n, oh, ow, cout, round_up(cout, 8) if out_mode != OUT_NCHW_F32 else cout)
        assert (out_geom.h, out_geom.w) == (oh, ow), (out_geom, oh, ow)
        d.out = out_geom.c_struct()
        self.desc = d
        self.in_geom, self.out_geom, self.out_mode = in_geom, out_geom, out_mode
        self.cout = cout
        info = _lib.ConvInfo()
        check(lib.hfc_conv_query(ctypes.byref(d), ctypes.byref(info)), "conv_query")
        self.info = info
        self.flops = info.flops
        self._packed = None
        self._packed_key = None
        self._packed_src = None

    def widenorm_supported(self):
        """True if this conv (NHWC fp16 output geometry, 768 < cout <= 1024) can run fused with the ChannelNorm that
        follows it through hfc_conv_forward_widenorm (host-side check)."""
        d = _lib.ConvDesc.from_buffer_copy(self.desc)
        d.norm = 1
        return lib.hfc_conv_widenorm_supported(ctypes.byref(d)) == 0

    def call_widenorm(self, x_act, weight, bias, gamma, beta, res1=None, res2=None, out_f32=None, out_act=None):
        """conv + bias + ChannelNorm over the whole (wide) channel row + activation [+ res1] [+ res2] in ONE launch:
        fp32 rows into `out_f32` (pitch = its row length) and / or the bordered fp16 buffer `out_act` (self.out_geom)."""
        assert x_act.is_cuda and x_act.dtype == torch.float16 and tuple(x_act.shape) == self.in_geom.shape
        assert self.out_mode == OUT_NHWC_F16 and (out_f32 is not None or out_act is not None)
        packed = self.packed_weights(weight)
        d = _lib.ConvDesc.from_buffer_copy(self.desc)
        d.norm = 1
        ld_res = 0
        for r in (res1, res2):
            if r is not None:
                assert r.dtype == torch.float32 and r.is_contiguous()
                ld_res = r.shape[-1]
        assert res1 is None or res2 is None or res1.shape[-1] == res2.shape[-1]
        if out_act is not None:
            assert tuple(out_act.shape) == self.out_geom.shape and out_act.dtype == torch.float16
        check(lib.hfc_conv_forward_widenorm(ctypes.byref(d), _ptr(x_act), _ptr(packed),
                                            _ptr(bias.detach().reshape(-1) if bias is not None else None),
                                            _ptr(gamma.detach().reshape(-1)), _ptr(beta.detach().reshape(-1)),
                                            _ptr(res1), _ptr(res2), ld_res, _ptr(out_f32),
                                            out_f32.shape[-1] if out_f32 is not None else 0, _ptr(out_act), _stream()),
              "conv_forward_widenorm")
        return out_act, out_f32

    def alloc_out(self, device):
        g = self.out_geom
        if self.out_mode == OUT_NHWC_F16:
            return g.alloc(device)
        if self.out_mode == OUT_NHWC_F32:
            return torch.empty((g.n * g.h * g.w, g.cpad), dtype=torch.float32, device=device)
        return torch.empty((g.n, self.cout, g.h, g.w), dtype=torch.float32, device=device)

    def packed_weights(self, weight, scale=None, scale_key=None):
        """scale: optional device scalar multiplied into every weight while packing (spectral norm's 1/sigma);
        scale_key: anything hashable that changes whenever the scale value may have changed."""
        key = (weight.data_ptr(), weight._version, weight.device, scale_key)
        if self._packed is None or self._packed_key != key:
            w = weight.detach()
            assert w.is_cuda and w.dtype == torch.float32 and w.is_contiguous()
            if self._packed is None or self._packed.device != w.device:
                self._packed = torch.empty(self.info.packed_weight_bytes // 2, dtype=torch.float16, device=w.device)
            if scale is None:
                check(lib.hfc_conv_pack_weights(ctypes.byref(self.desc), _ptr(w), _ptr(self._packed), _stream()),
                      "conv_pack_weights")
            else:
                check(lib.hfc_conv_pack_weights_scaled(ctypes.byref(self.desc), _ptr(w), _ptr(scale),
                                                       _ptr(self._packed), _stream()), "conv_pack_weights_scaled")
            self._packed_key = key
            # keep the source storage alive: a NEW tensor can then never reuse this address (caching allocator) with
            # the same version counter and be mistaken for the packed one
            self._packed_src = weight.detach()
        return self._packed

    def __call__(self, x_act, weight, bias=None, gamma=None, beta=None, out=None, scale=None, scale_key=None):
        assert x_act.is_cuda and x_act.dtype == torch.float16 and tuple(x_act.shape) == self.in_geom.shape, \
            (tuple(x_act.shape), self.in_geom.shape)
        packed = self.packed_weights(weight, scale, scale_key)
        if out is None:
            out = self.alloc_out(x_act.device)
        b = bias.detach().reshape(-1) if bias is not None else None
        g = gamma.detach().reshape(-1) if gamma is not None else None
        bt = beta.detach().reshape(-1) if beta is not None else None
        check(lib.hfc_conv_forward(ctypes.byref(self.desc), _ptr(x_act), _ptr(packed), _ptr(b), _ptr(g),
                                   _ptr(bt), _ptr(out), _stream()), "conv_forward")
        return out


def latent_likelihood(y, mean, scale_raw, noise=None, scale_lower_bound=0.11, likelihood_type="gaussian", sums=None):
    """Fused conditional likelihood; returns (decoded, sums) with sums = [sum log p_noisy, sum log p_quant]
    (natural log, fp64, on device)."""
    for t in (y, mean, scale_raw) + ((noise,) if noise is not None else ()):
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == y.shape
    decoded = torch.empty_like(y)
    if sums is None:
        sums = torch.zeros(2, dtype=torch.float64, device=y.device)   # else: caller-provided, already zeroed
    lt = {"gaussian": 0, "logistic": 1}[likelihood_type]
    check(lib.hfc_latent_likelihood(_ptr(y), _ptr(mean), _ptr(scale_raw), _ptr(noise), y.numel(),
                                    float(scale_lower_bound), lt, _ptr(decoded), _ptr(sums), _stream()),
          "latent_likelihood")
    return decoded, sums


def pack_density_params(Hs, a_s, bs):
    """(H_k, a_k, b_k), k=0..3, shapes (C,f_{k+1},f_k)/(C,f_{k+1},1) -> (C, 64) fp32 rows in the order
    the kernel expects: softplus(H_k) row-major, b_k, tanh(a_k) per layer."""
    C = Hs[0].shape[0]
    parts = []
    for H, a, b in zip(Hs, a_s, bs):
        parts += [torch.nn.functional.softplus(H.detach()).reshape(C, -1), b.detach().reshape(C, -1),
                  torch.tanh(a.detach()).reshape(C, -1)]
    p = torch.cat(parts, dim=1)
    assert p.shape[1] == 44, p.shape
    out = torch.zeros((C, 64), dtype=torch.float32, device=p.device)
    out[:, :44] = p
    return out.contiguous()


def hyperlatent_likelihood(z, params64, noise=None, sums=None):
    """Factorized-density likelihood of z at z+noise and round(z). Returns (z_noisy|None, z_quant, sums)."""
    assert z.is_cuda and z.dtype == torch.float32 and z.is_contiguous() and z.dim() == 4
    n, c, h, w = z.shape
    assert tuple(params64.shape) == (c, 64) and params64.is_contiguous()
    z_quant = torch.empty_like(z)
    z_noisy = torch.empty_like(z) if noise is not None else None
    if sums is None:
        sums = torch.zeros(2, dtype=torch.float64, device=z.device)
    check(lib.hfc_hyperlatent_likelihood(_ptr(z), _ptr(noise), _ptr(params64), n, c, h * w, _ptr(z_noisy),
                                         _ptr(z_quant), _ptr(sums), _stream()), "hyperlatent_likelihood")
    return z_noisy, z_quant, sums


def disc_input(x, ctx_act, ctx_geom, out_geom, scale, out=None):
    """cat(x, nearest-upsample(ctx)) -> bordered act buffer (Discriminator.forward, discriminator.py:75-79)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
    if out is None:
        out = out_geom.alloc(x.device)
    cg, og = ctx_geom.c_struct(), out_geom.c_struct()
    check(lib.hfc_disc_input(_ptr(x), x.shape[1], _ptr(ctx_act), ctypes.byref(cg), scale, ctypes.byref(og), _ptr(out),
                             _stream()), "disc_input")
    return out


def spectral_sigma(weight_orig, u, v, power_iteration, workspace=None):
    """torch.nn.utils.spectral_norm's sigma for `weight_orig` (cout, ...) with buffers u, v (updated in place when
    power_iteration).  Returns (sigma, inv_sigma) device scalars."""
    w = weight_orig.detach()
    rows, cols = w.shape[0], w.numel() // w.shape[0]
    assert w.is_contiguous() and u.numel() == rows and v.numel() == cols
    if workspace is None:
        workspace = torch.empty(rows + cols, dtype=torch.float32, device=w.device)
    out = torch.empty(2, dtype=torch.float32, device=w.device)
    check(lib.hfc_spectral_sigma(_ptr(w), rows, cols, _ptr(u), _ptr(v), int(power_iteration), _ptr(workspace),
                                 _ptr(out[0:1]), _ptr(out[1:2]), _stream()), "spectral_sigma")
    return out[0], out[1:2]


def gan_sums(logits):
    """[sum BCE(real,1), sum BCE(gen,0), sum BCE(gen,1), sum sigmoid(real), sum sigmoid(gen)] (fp64, device)."""
    lg = logits.reshape(-1)
    assert lg.is_cuda and lg.dtype == torch.float32 and lg.is_contiguous() and lg.numel() % 2 == 0
    sums = torch.zeros(5, dtype=torch.float64, device=lg.device)
    check(lib.hfc_gan_sums(_ptr(lg), lg.numel() // 2, _ptr(sums), _stream()), "gan_sums")
    return sums


def sqdiff_sum(a, b, scale=255.0):
    assert a.shape == b.shape and a.is_cuda and a.dtype == torch.float32 and a.is_contiguous() and b.is_contiguous()
    out = torch.zeros(1, dtype=torch.float64, device=a.device)
    check(lib.hfc_sqdiff_sum(_ptr(a), _ptr(b), a.numel(), float(scale), _ptr(out), _stream()), "sqdiff_sum")
    return out[0]


def lpips_layer(f0, f1, lin_w, out):
    """out[i] += spatial mean of the LIN-weighted squared distance between channel-normalised features."""
    assert f0.shape == f1.shape and f0.is_cuda and f0.dtype == torch.float32
    f0, f1 = f0.contiguous(), f1.contiguous()
    n, c, h, w = f0.shape
    lw = lin_w.reshape(-1).contiguous()
    assert lw.numel() == c and out.numel() == n and out.dtype == torch.float32
    check(lib.hfc_lpips_layer(_ptr(f0), _ptr(f1), _ptr(lw), n, c, h * w, _ptr(out), _stream()), "lpips_layer")
    return out


# ------------------------------------------------------------------------------------------------------------
# autograd wrappers of the fused elementwise kernels (training path)
# ------------------------------------------------------------------------------------------------------------
class LatentLikelihoodFn(torch.autograd.Function):
    """(y, mean, scale_raw, noise) -> (decoded, sums[2]); gradient flows through decoded (straight-through to y)
    and sums[0] (the noisy log-likelihood sum); sums[1] is consumed via .item() in the reference (losses.py:21)."""

    @staticmethod
    def forward(ctx, y, mean, scale_raw, noise, lb, kind):
        decoded, sums = latent_likelihood(y, mean, scale_raw, noise, lb, kind)
        ctx.save_for_backward(y, mean, scale_raw, noise)
        ctx.lb, ctx.kind = lb, kind
        return decoded, sums

    @staticmethod
    def backward(ctx, d_decoded, d_sums):
        y, mean, scale_raw, noise = ctx.saved_tensors
        dy, dm, ds = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
        g = d_sums[0:1].to(torch.float32).contiguous() if d_sums is not None else torch.zeros(1, device=y.device)
        dd = d_decoded.contiguous() if d_decoded is not None else None
        lt = {"gaussian": 0, "logistic": 1}[ctx.kind]
        check(lib.hfc_latent_likelihood_bwd(_ptr(y), _ptr(mean), _ptr(scale_raw), _ptr(noise), _ptr(dd), _ptr(g), 1.0,
                                            y.numel(), float(ctx.lb), lt, _ptr(dy), _ptr(dm), _ptr(ds), _stream()),
              "latent_likelihood_bwd")
        return dy, dm, ds, None, None, None


class HyperlatentLikelihoodFn(torch.autograd.Function):
    """(z, packed_params, noise) -> (z_noisy, z_quant, sums[2]); gradient through z_noisy and sums[0]."""

    @staticmethod
    def forward(ctx, z, params64, noise):
        z_noisy, z_quant, sums = hyperlatent_likelihood(z, params64, noise)
        ctx.save_for_backward(z_noisy, params64)
        ctx.mark_non_differentiable(z_quant)
        return z_noisy, z_quant, sums

    @staticmethod
    def backward(ctx, d_noisy, d_quant, d_sums):
        z_noisy, params64 = ctx.saved_tensors
        n, c, h, w = z_noisy.shape
        dz = torch.empty_like(z_noisy)
        dp = torch.empty_like(params64)
        g = d_sums[0:1].to(torch.float32).contiguous() if d_sums is not None else torch.zeros(1, device=dz.device)
        dn = d_noisy.contiguous() if d_noisy is not None else None
        check(lib.hfc_hyperlatent_likelihood_bwd(_ptr(z_noisy), _ptr(dn), _ptr(params64), _ptr(g), 1.0, n, c, h * w,
                                                 _ptr(dz), _ptr(dp), _stream()), "hyperlatent_likelihood_bwd")
        return dz, dp, None


def pack_density_params_autograd(Hs, a_s, bs):
    """Differentiable version of pack_density_params (14 080 scalars: plain torch ops carry the chain rule back to
    H_k, a_k, b_k)."""
    C = Hs[0].shape[0]
    parts = []
    for H, a, b in zip(Hs, a_s, bs):
        parts += [torch.nn.functional.softplus(H).reshape(C, -1), b.reshape(C, -1), torch.tanh(a).reshape(C, -1)]
    p = torch.cat(parts, dim=1)
    return torch.nn.functional.pad(p, (0, 64 - p.shape[1])).contiguous()


class LpipsLayerFn(torch.autograd.Function):
    """per-image LPIPS distance of one trunk layer; gradient w.r.t. f1 (the reconstruction's features) only."""

    @staticmethod
    def forward(ctx, f0, f1, lin_w):
        f0, f1 = f0.contiguous(), f1.contiguous()
        out = torch.zeros(f0.shape[0], dtype=torch.float32, device=f0.device)
        lpips_layer(f0, f1, lin_w, out)
        ctx.save_for_backward(f0, f1, lin_w)
        return out

    @staticmethod
    def backward(ctx, d_out):
        f0, f1, lin_w = ctx.saved_tensors
        n, c, h, w = f1.shape
        df1 = torch.empty_like(f1)
        check(lib.hfc_lpips_layer_bwd(_ptr(f0), _ptr(f1), _ptr(lin_w.reshape(-1).contiguous()), _ptr(d_out.contiguous()),
                                      n, c, h * w, _ptr(df1), _stream()), "lpips_layer_bwd")
        return None, df1, None


class SqDiffMeanFn(torch.autograd.Function):
    """mean((s*a - s*b)^2) with gradient w.r.t. a (src/model.py:190-194)."""

    @staticmethod
    def forward(ctx, a, b, scale):
        a, b = a.contiguous(), b.contiguous()
        ctx.save_for_backward(a, b)
        ctx.scale = scale
        return (sqdiff_sum(a, b, scale) / a.numel()).to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        return (a - b) * (g * (2.0 * ctx.scale * ctx.scale / a.numel())), None, None


class GanLossFn(torch.autograd.Function):
    """Non-saturating GAN losses (src/loss/losses.py:30-41) on [real, gen] logits: mode 0 = generator loss
    mean BCE(gen, 1), mode 1 = discriminator loss mean BCE(real, 1) + mean BCE(gen, 0)."""

    @staticmethod
    def forward(ctx, logits_real, logits_gen, mode):
        lg = torch.cat([logits_real.reshape(-1), logits_gen.reshape(-1)]).contiguous()
        ctx.save_for_backward(lg)
        ctx.mode, ctx.shapes = mode, (logits_real.shape, logits_gen.shape)
        sums = gan_sums(lg).to(torch.float32) / logits_real.numel()
        return sums[0] + sums[1] if mode == 1 else sums[2]

    @staticmethod
    def backward(ctx, g):
        lg, = ctx.saved_tensors
        half = lg.numel() // 2
        out = torch.empty_like(lg)
        g = g.to(torch.float32).contiguous()
        check(lib.hfc_gan_grad(_ptr(lg), half, ctx.mode, _ptr(g), _ptr(out), _stream()), "gan_grad")
        return out[:half].view(ctx.shapes[0]), out[half:].view(ctx.shapes[1]), None


# ------------------------------------------------------------------------------------------------------------
# compress / decompress path: the GPU half either side of the host rANS coder (csrc/symbols.cu)
# ------------------------------------------------------------------------------------------------------------
_TABLE_CACHE = {}


def _scale_table(scale_table, device):
    """Device copy of the scale table + whether it is non-decreasing (then the kernels binary-search it); cached per
    (storage, version, device) so the check and the copy cost nothing per call."""
    key = (scale_table.data_ptr(), scale_table._version, scale_table.device, device)
    hit = _TABLE_CACHE.get(key)
    if hit is None:
        host = scale_table.detach().to(dtype=torch.float32, device="cpu").reshape(-1)
        is_sorted = int(bool((host[1:] >= host[:-1]).all()))
        hit = (scale_table.detach().to(device=device, dtype=torch.float32).contiguous(), is_sorted, scale_table)
        if len(_TABLE_CACHE) > 16:
            _TABLE_CACHE.clear()
        _TABLE_CACHE[key] = hit
    return hit[0], hit[1]


def quantize_symbols(x, mean=None, scale_raw=None, scale_table=None, scale_lower_bound=0.11,
                     likelihood_type="gaussian", layout=_lib.SYM_BATCH_STEPS, want_symbols=True, want_indices=True,
                     want_dequant=False, want_bits=False):
    """One pass over the (N, C, H, W) latents: int32 symbols floor(x + .5 - mean) and table indices in coder order
    (`layout`), optionally the dequantised latents (NCHW fp32) and the natural-log likelihood sum of the quantised
    values (fp64 device scalar).  Returns a dict with the requested entries."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4
    for t in (mean, scale_raw):
        assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == x.shape)
    n, c, h, w = x.shape
    dev = x.device
    out = {}
    if want_symbols:
        out["symbols"] = torch.empty(n * c * h * w, dtype=torch.int32, device=dev)
    if want_indices:
        out["indices"] = torch.empty(n * c * h * w, dtype=torch.int32, device=dev)
    if want_dequant:
        out["dequant"] = torch.empty_like(x)
    if want_bits:
        assert scale_raw is not None
        out["bits_sum"] = torch.zeros(1, dtype=torch.float64, device=dev)
    tbl, is_sorted = None, 0
    if scale_raw is not None:
        tbl, is_sorted = _scale_table(scale_table, dev)
    lt = {"gaussian": 0, "logistic": 1}[likelihood_type]
    check(lib.hfc_quantize_symbols(_ptr(x), _ptr(mean), _ptr(scale_raw), n, c, h * w, _ptr(tbl),
                                   tbl.numel() if tbl is not None else 0, float(scale_lower_bound), lt, int(layout),
                                   is_sorted, _ptr(out.get("symbols")), _ptr(out.get("indices")), _ptr(out.get("dequant")),
                                   _ptr(out.get("bits_sum")), _stream()), "quantize_symbols")
    if want_bits:
        out["bits_sum"] = out["bits_sum"][0]
    return out


def scale_indices(scale_raw, scale_table, scale_lower_bound=0.11, layout=_lib.SYM_BATCH_STEPS):
    """Table index of every scale (PriorEntropyModel.compute_indices) as flat int32 in coder order."""
    assert scale_raw.is_cuda and scale_raw.dtype == torch.float32 and scale_raw.is_contiguous() and scale_raw.dim() == 4
    n, c, h, w = scale_raw.shape
    tbl, is_sorted = _scale_table(scale_table, scale_raw.device)
    out = torch.empty(n * c * h * w, dtype=torch.int32, device=scale_raw.device)
    check(lib.hfc_scale_indices(_ptr(scale_raw), n, c, h * w, _ptr(tbl), tbl.numel(), float(scale_lower_bound),
                                int(layout), is_sorted, _ptr(out), _stream()), "scale_indices")
    return out


def dequantize_symbols(symbols, mean, shape, layout=_lib.SYM_BATCH_STEPS):
    """int32 symbols in coder order (+ NCHW fp32 mean, may be None) -> NCHW fp32 latents."""
    n, c, h, w = shape
    assert symbols.is_cuda and symbols.dtype == torch.int32 and symbols.is_contiguous() and symbols.numel() == n * c * h * w
    assert mean is None or (mean.is_cuda and mean.dtype == torch.float32 and mean.is_contiguous()
                            and tuple(mean.shape) == tuple(shape))
    out = torch.empty(shape, dtype=torch.float32, device=symbols.device)
    check(lib.hfc_dequantize_symbols(_ptr(symbols), _ptr(mean), n, c, h * w, int(layout), _ptr(out), _stream()),
          "dequantize_symbols")
    return out


# ------------------------------------------------------------------------------------------------------------
# LPIPS trunk pieces in the activation format (csrc/lpips_trunk.cu)
# ------------------------------------------------------------------------------------------------------------
def lpips_prep(target, pred, geom, normalize, shift, scale, out=None):
    """(n, 3, h, w) target / pred -> (2n, hs, ws, 64) fp16 scaled space-to-depth buffer `geom` (n = 2n images)."""
    assert target.shape == pred.shape and target.is_cuda and pred.is_cuda
    target, pred = target.contiguous(), pred.contiguous()
    n, c, h, w = target.shape
    assert c == 3 and geom.n == 2 * n and geom.cpad == 64
    if out is None:
        out = geom.alloc(target.device)
    check(lib.hfc_lpips_prep(_ptr(target), _ptr(pred), n, h, w, geom.h, geom.w, int(bool(normalize)),
                             _ptr(shift.reshape(-1).contiguous()), _ptr(scale.reshape(-1).contiguous()), _ptr(out),
                             _stream()), "lpips_prep")
    return out


def lpips_prep_bwd(g_rows, n, h, w, hs, ws, normalize, scale):
    assert g_rows.dtype == torch.float32 and g_rows.is_contiguous() and g_rows.shape[0] == n * hs * ws
    dpred = torch.empty((n, 3, h, w), dtype=torch.float32, device=g_rows.device)
    check(lib.hfc_lpips_prep_bwd(_ptr(g_rows), g_rows.shape[1], n, h, w, hs, ws, int(bool(normalize)),
                                 _ptr(scale.reshape(-1).contiguous()), _ptr(dpred), _stream()), "lpips_prep_bwd")
    return dpred


def maxpool3s2(x_act, geom, out_geom, out=None):
    """nn.MaxPool2d(3, 2) on a border-less NHWC fp16 buffer."""
    assert tuple(x_act.shape) == geom.shape and x_act.dtype == torch.float16
    assert (out_geom.h, out_geom.w) == ((geom.h - 3) // 2 + 1, (geom.w - 3) // 2 + 1) and out_geom.cpad == geom.cpad
    if out is None:
        out = out_geom.alloc(x_act.device)
    g = geom.c_struct()
    check(lib.hfc_maxpool3s2(_ptr(x_act), ctypes.byref(g), _ptr(out), _stream()), "maxpool3s2")
    return out


def maxpool3s2_bwd(g_out_rows, x_act, geom):
    """Adjoint of maxpool3s2 for the images described by `geom` (x_act = the pooled layer's input for those images):
    fp32 rows [n*oh*ow][ld] -> fp32 rows [n*h*w][c]."""
    assert g_out_rows.dtype == torch.float32 and g_out_rows.is_contiguous() and x_act.dtype == torch.float16
    g_in = torch.zeros((geom.n * geom.h * geom.w, geom.c), dtype=torch.float32, device=g_out_rows.device)
    g = geom.c_struct()
    check(lib.hfc_maxpool3s2_bwd(_ptr(g_out_rows), g_out_rows.shape[1], _ptr(x_act), ctypes.byref(g), _ptr(g_in),
                                 g_in.shape[1], _stream()), "maxpool3s2_bwd")
    return g_in


def lpips_nhwc(feat_act, geom, lin_w, out):
    """out[i] += LPIPS distance of one layer; feat_act (2n, h, w, cpad) holds target [0, n) and reconstruction [n, 2n)."""
    assert tuple(feat_act.shape) == geom.shape and geom.n % 2 == 0 and out.numel() == geom.n // 2
    check(lib.hfc_lpips_nhwc(_ptr(feat_act), geom.n // 2, geom.h * geom.w, geom.c, geom.cpad,
                             _ptr(lin_w.reshape(-1).contiguous()), _ptr(out), _stream()), "lpips_nhwc")
    return out


def lpips_nhwc_bwd(feat_act, geom, lin_w, upstream, g_in_rows=None):
    """fp32 rows [n*h*w][c]: gradient w.r.t. the pre-ReLU features of the reconstruction half (see hfc.h)."""
    n = geom.n // 2
    out = torch.empty((n * geom.h * geom.w, geom.c), dtype=torch.float32, device=feat_act.device)
    assert g_in_rows is None or (g_in_rows.dtype == torch.float32 and g_in_rows.is_contiguous()
                                 and g_in_rows.shape[0] == out.shape[0])
    check(lib.hfc_lpips_nhwc_bwd(_ptr(feat_act), n, geom.h * geom.w, geom.c, geom.cpad,
                                 _ptr(lin_w.reshape(-1).contiguous()), _ptr(upstream.contiguous()), _ptr(g_in_rows),
                                 g_in_rows.shape[1] if g_in_rows is not None else 0, _ptr(out), out.shape[1], _stream()),
          "lpips_nhwc_bwd")
    return out


# ------------------------------------------------------------------------------------------------------------
# discretised mixture likelihood of the latents (csrc/dlmm.cu; HyperpriorDLMM, src/hyperprior.py:340-458)
# ------------------------------------------------------------------------------------------------------------
def dlmm_likelihood(x, dlmm_params, noise=None, likelihood_type="gaussian", straight_through=True, sums=None):
    """x (N, C, H, W), dlmm_params (N, 3*C*K, H, W) -> (decoded, sums[2]) with sums = [sum L(x + noise), sum L(round x)]
    (natural log, fp64, on device)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4
    n, c, h, w = x.shape
    assert dlmm_params.is_cuda and dlmm_params.dtype == torch.float32 and dlmm_params.is_contiguous()
    assert dlmm_params.shape[0] == n and tuple(dlmm_params.shape[2:]) == (h, w) and dlmm_params.shape[1] % (3 * c) == 0
    k = dlmm_params.shape[1] // (3 * c)
    assert noise is None or (noise.is_cuda and noise.is_contiguous() and noise.shape == x.shape)
    decoded = torch.empty_like(x)
    if sums is None:
        sums = torch.zeros(2, dtype=torch.float64, device=x.device)
    lt = {"gaussian": 0, "logistic": 1}[likelihood_type]
    check(lib.hfc_dlmm_likelihood(_ptr(x), _ptr(noise), _ptr(dlmm_params), n, c, k, h * w, lt, int(bool(straight_through)),
                                  _ptr(decoded), _ptr(sums), _stream()), "dlmm_likelihood")
    return decoded, sums


def dlmm_likelihood_bwd(x, dlmm_params, noise, d_decoded, g_nbpp, likelihood_type="gaussian"):
    n, c, h, w = x.shape
    k = dlmm_params.shape[1] // (3 * c)
    dx, dparams = torch.empty_like(x), torch.empty_like(dlmm_params)
    lt = {"gaussian": 0, "logistic": 1}[likelihood_type]
    check(lib.hfc_dlmm_likelihood_bwd(_ptr(x), _ptr(noise), _ptr(dlmm_params), _ptr(d_decoded), _ptr(g_nbpp), 1.0, n, c,
                                      k, h * w, lt, _ptr(dx), _ptr(dparams), _stream()), "dlmm_likelihood_bwd")
    return dx, dparams


class DlmmLikelihoodFn(torch.autograd.Function):
    """(x, dlmm_params, noise) -> (decoded, sums[2]); gradient through decoded (straight-through to x) and sums[0]."""

    @staticmethod
    def forward(ctx, x, dlmm_params, noise, kind, straight_through):
        decoded, sums = dlmm_likelihood(x, dlmm_params, noise, kind, straight_through)
        ctx.save_for_backward(x, dlmm_params, noise)
        ctx.kind = kind
        return decoded, sums

    @staticmethod
    def backward(ctx, d_decoded, d_sums):
        x, dlmm_params, noise = ctx.saved_tensors
        g = d_sums[0:1].to(torch.float32).contiguous() if d_sums is not None else torch.zeros(1, device=x.device)
        dd = d_decoded.contiguous() if d_decoded is not None else None
        dx, dparams = dlmm_likelihood_bwd(x, dlmm_params, noise, dd, g, ctx.kind)
        return dx, dparams, None, None, None


# ------------------------------------------------------------------------------------------------------------
# PSNR / SSIM / MS-SSIM of the evaluation loop (csrc/ssim.cu; src/helpers/metrics.py)
# ------------------------------------------------------------------------------------------------------------
_metrics_ws_cache = {}


def _metrics_ws(key, need, device):
    """Scratch of the metric kernels, one buffer per (kind, device), grown on demand; the launches that use it are ordered
    on the current stream."""
    if need < 0:
        raise _lib.HfcError(f"libhfc {key} workspace query failed: {lib.hfc_last_error().decode('utf-8', 'replace')}")
    buf = _metrics_ws_cache.get((key, device))
    if buf is None or buf.numel() * 8 < need:
        buf = _metrics_ws_cache[(key, device)] = torch.empty(max(1, (need + 7) // 8), dtype=torch.float64, device=device)
    return buf, buf.numel() * 8


def _ssim_forward_launches(x, y, taps, c1, c2, weights, relu_last, size_average, ws, ws_bytes):
    """The level and finalize launches of ssim_levels on workspace `ws`.  Returns (out, pyramid): pyramid[l] is level l's
    input pair (x, y at level 0, then the pooled planes the level kernels wrote)."""
    n, c, h, w = x.shape
    win = taps.shape[-1]
    levels = len(weights)
    pyramid = []
    for level in range(levels):
        pyramid.append((x, y))
        if level < levels - 1:
            hp, wp = (x.shape[2] + 1) // 2, (x.shape[3] + 1) // 2
            px = torch.empty((n, c, hp, wp), dtype=torch.float32, device=x.device)
            py = torch.empty_like(px)
        else:
            px = py = None
        check(lib.hfc_ssim_level(_ptr(x), _ptr(y), n, c, h, w, level, _ptr(taps), win, c1, c2, _ptr(px), _ptr(py),
                                 _ptr(ws), ws_bytes, _stream()), "ssim_level")
        x, y = px, py
    out = torch.empty(1 if size_average else n, dtype=torch.float32, device=ws.device)
    wts = (ctypes.c_float * levels)(*weights)
    check(lib.hfc_ssim_finalize(n, c, h, w, win, levels, wts, int(bool(relu_last)), int(bool(size_average)), _ptr(ws),
                                ws_bytes, _ptr(out), _stream()), "ssim_finalize")
    return (out.reshape(()) if size_average else out), pyramid


def _ssim_backward_launches(pyramid, taps, c1, c2, weights, relu_last, size_average, ws, ws_bytes, grad_out, need_x,
                            need_y):
    """Gradients of ssim_levels' output w.r.t. pyramid[0] from the forward's workspace (its per-plane level sums) and
    the kept pyramid: one coefficient launch, then per level (coarsest first) a gradient-map and a level-backward launch.
    Returns (dx, dy), None where not needed."""
    x, y = pyramid[0]
    n, c, h, w = x.shape
    win = taps.shape[-1]
    levels = len(weights)
    dev = x.device
    g = grad_out.to(dtype=torch.float32).contiguous()
    coef = torch.empty(n * c * levels * 2, dtype=torch.float32, device=dev)
    wts = (ctypes.c_float * levels)(*weights)
    check(lib.hfc_ssim_grad_coeffs(n, c, h, w, win, levels, wts, int(bool(relu_last)), int(bool(size_average)), _ptr(ws),
                                   ws_bytes, _ptr(g), _ptr(coef), _stream()), "ssim_grad_coeffs")
    maps_bytes = int(lib.hfc_ssim_grad_maps_bytes(n, c, h, w, win, levels))
    if maps_bytes < 0:
        raise _lib.HfcError(f"libhfc ssim_grad_maps_bytes failed: {lib.hfc_last_error().decode('utf-8', 'replace')}")
    maps = torch.empty(max(4, maps_bytes // 4), dtype=torch.float32, device=dev)
    dx = dy = None
    for level in reversed(range(levels)):
        xl, yl = pyramid[level]
        check(lib.hfc_ssim_grad_maps(_ptr(xl), _ptr(yl), n, c, h, w, level, levels, _ptr(taps), win, c1, c2, _ptr(coef),
                                     _ptr(maps), maps.numel() * 4, _stream()), "ssim_grad_maps")
        gx = torch.empty_like(xl) if need_x else None
        gy = torch.empty_like(yl) if need_y else None
        check(lib.hfc_ssim_level_bwd(_ptr(xl), _ptr(yl), _ptr(maps), n, c, h, w, level, _ptr(taps), win, _ptr(dx),
                                     _ptr(dy), _ptr(gx), _ptr(gy), _stream()), "ssim_level_bwd")
        dx, dy = gx, gy
    return dx, dy


def _ssim_check_args(x, y, taps):
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and y.shape == x.shape and y.dtype == x.dtype
    win = taps.shape[-1]
    assert taps.is_cuda and taps.dtype == torch.float32 and taps.is_contiguous() and tuple(taps.shape) == (x.shape[1], win)


def ssim_levels(x, y, taps, c1, c2, weights, relu_last, size_average):
    """x, y (N, C, H, W) fp32 CUDA; taps (C, win) fp32 on x's device.  len(weights) SSIM levels (2x2 average pool in
    between) -> prod_l value_l ** weights[l] per plane, averaged over (N, C) (0-d tensor) or over C per image ((N,)).
    len(weights) + 1 launches, no synchronisation."""
    _ssim_check_args(x, y, taps)
    x, y = x.contiguous(), y.contiguous()
    n, c, h, w = x.shape
    ws, ws_bytes = _metrics_ws("ssim", int(lib.hfc_ssim_ws_bytes(n, c, h, w, taps.shape[-1], len(weights))), x.device)
    return _ssim_forward_launches(x, y, taps, c1, c2, weights, relu_last, size_average, ws, ws_bytes)[0]


class SsimLevelsFn(torch.autograd.Function):
    """ssim_levels with a gradient w.r.t. x and y.  The forward runs ssim_levels' launches (bit-identical values) on a
    workspace of its own, so that a second forward before this one's backward cannot overwrite the per-plane level sums
    the backward reads; it keeps the pooled pyramid.  taps, c1, c2, weights and the flags are constants."""

    @staticmethod
    def forward(ctx, x, y, taps, c1, c2, weights, relu_last, size_average):
        _ssim_check_args(x, y, taps)
        xc, yc = x.contiguous(), y.contiguous()
        n, c, h, w = xc.shape
        need = int(lib.hfc_ssim_ws_bytes(n, c, h, w, taps.shape[-1], len(weights)))
        if need < 0:
            raise _lib.HfcError(f"libhfc ssim workspace query failed: {lib.hfc_last_error().decode('utf-8', 'replace')}")
        ws = torch.empty(max(1, (need + 7) // 8), dtype=torch.float64, device=xc.device)
        out, pyramid = _ssim_forward_launches(xc, yc, taps, c1, c2, weights, relu_last, size_average, ws, ws.numel() * 8)
        ctx.save_for_backward(x, y)
        ctx.pooled = pyramid[1:]
        ctx.ws = ws
        ctx.consts = (taps, c1, c2, list(weights), relu_last, size_average)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        need_x, need_y = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_x or need_y):
            return (None,) * 8
        x, y = ctx.saved_tensors
        taps, c1, c2, weights, relu_last, size_average = ctx.consts
        pyramid = [(x.contiguous(), y.contiguous())] + ctx.pooled
        dx, dy = _ssim_backward_launches(pyramid, taps, c1, c2, weights, relu_last, size_average, ctx.ws,
                                         ctx.ws.numel() * 8, grad_out, need_x, need_y)
        return dx, dy, None, None, None, None, None, None


def ssim_levels_grad(x, y, taps, c1, c2, weights, relu_last, size_average):
    """ssim_levels, differentiable w.r.t. x and y when grad mode is on and either requires a gradient (SsimLevelsFn);
    otherwise ssim_levels itself.  Backward: at most 2 * len(weights) + 1 launches, no synchronisation."""
    if torch.is_grad_enabled() and (x.requires_grad or y.requires_grad):
        return SsimLevelsFn.apply(x, y, taps, c1, c2, list(weights), relu_last, size_average)
    return ssim_levels(x, y, taps, c1, c2, weights, relu_last, size_average)


def psnr(a, b, max_val=255.0):
    """a, b (N, ...) fp32 CUDA -> (N,) float64 per-image PSNR in dB (2 launches, no synchronisation)."""
    assert a.is_cuda and a.dtype == torch.float32 and b.shape == a.shape and b.dtype == a.dtype and a.dim() >= 1
    a, b = a.contiguous(), b.contiguous()
    n = a.shape[0]
    per_image = a.numel() // n
    ws, ws_bytes = _metrics_ws("psnr", int(lib.hfc_psnr_ws_bytes(n, per_image)), a.device)
    out = torch.empty(n, dtype=torch.float64, device=a.device)
    check(lib.hfc_psnr(_ptr(a), _ptr(b), n, per_image, float(max_val), _ptr(ws), ws_bytes, _ptr(out), _stream()), "psnr")
    return out
