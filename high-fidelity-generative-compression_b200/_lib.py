"""ctypes binding of libhfc.so (the C ABI declared in include/hfc.h).

There is no fallback: if the shared library is missing the import fails, and every compute entry
point returns an error (raised here as RuntimeError) on a machine without an sm_100 GPU.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HFC_LIB_PATH") or os.path.join(_HERE, "libhfc.so")   # override: A/B builds
CSRC_DIR = os.path.join(_HERE, "csrc")


class ActGeom(ctypes.Structure):
    """Mirror of ``hfc_act_geom``."""
    _fields_ = [(k, ctypes.c_int32) for k in ("n", "h", "w", "c", "cpad", "pt", "pl", "pb", "pr")]


class ConvDesc(ctypes.Structure):
    """Mirror of ``hfc_conv_desc``."""
    _fields_ = [
        ("inp", ActGeom),
        ("kh", ctypes.c_int32), ("kw", ctypes.c_int32),
        ("stride", ctypes.c_int32), ("transposed", ctypes.c_int32),
        ("pad_mode", ctypes.c_int32),
        ("pad_t", ctypes.c_int32), ("pad_l", ctypes.c_int32),
        ("pad_b", ctypes.c_int32), ("pad_r", ctypes.c_int32),
        ("cout", ctypes.c_int32), ("window", ctypes.c_int32),
        ("out_mode", ctypes.c_int32),
        ("out", ActGeom),
        ("out_reflect", ctypes.c_int32),
        ("act", ctypes.c_int32), ("norm", ctypes.c_int32),
        ("eps", ctypes.c_float),
        ("block_n", ctypes.c_int32), ("precision", ctypes.c_int32),
        ("cluster_m", ctypes.c_int32), ("cluster_n", ctypes.c_int32),
        ("wide", ctypes.c_int32), ("a_bf16", ctypes.c_int32), ("b_bf16", ctypes.c_int32),
        ("dgrad", ctypes.c_int32), ("pair", ctypes.c_int32),
    ]


class WgradDesc(ctypes.Structure):
    """Mirror of ``hfc_wgrad_desc``."""
    _fields_ = [
        ("plain", ActGeom), ("shifted", ActGeom),
        ("ntaps", ctypes.c_int32), ("stride", ctypes.c_int32), ("bf16", ctypes.c_int32), ("k_splits", ctypes.c_int32),
        ("pair", ctypes.c_int32), ("window", ctypes.c_int32),
        ("tap_dh", ctypes.c_int8 * 64), ("tap_dw", ctypes.c_int8 * 64),
    ]


class ConvInfo(ctypes.Structure):
    """Mirror of ``hfc_conv_info``."""
    _fields_ = [
        ("packed_weight_bytes", ctypes.c_size_t),
        ("out_h", ctypes.c_int32), ("out_w", ctypes.c_int32), ("phases", ctypes.c_int32),
        ("block_n", ctypes.c_int32), ("n_tiles", ctypes.c_int32), ("m_tiles", ctypes.c_int32),
        ("stages", ctypes.c_int32), ("k_total", ctypes.c_int32),
        ("cluster_m", ctypes.c_int32), ("cluster_n", ctypes.c_int32), ("wide", ctypes.c_int32),
        ("pair", ctypes.c_int32), ("tapn", ctypes.c_int32), ("nsub", ctypes.c_int32),
        ("flops", ctypes.c_double),
    ]


PAD_ZERO, PAD_REFLECT = 0, 1
ACT_NONE, ACT_RELU, ACT_LEAKY02 = 0, 1, 2
OUT_NHWC_F16, OUT_NHWC_F32, OUT_NCHW_F32 = 0, 1, 2
PREC_F16, PREC_BF16X3 = 0, 1
SYM_BATCH_STEPS, SYM_PIXEL_STEPS = 0, 1

# name -> (restype, argtypes); doubles as the list of symbols the ABI test checks.
_vp, _i32, _i64, _f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
SIGNATURES = {
    "hfc_abi_version": (ctypes.c_int, []),
    "hfc_last_error": (ctypes.c_char_p, []),
    "hfc_device_info": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)] * 3),
    "hfc_launch_count": (ctypes.c_ulonglong, []),
    "hfc_conv_query": (ctypes.c_int, [ctypes.POINTER(ConvDesc), ctypes.POINTER(ConvInfo)]),
    "hfc_conv_pack_weights": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp]),
    "hfc_conv_pack_weights_scaled": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp]),
    "hfc_disc_input": (ctypes.c_int, [_vp, _i32, _vp, ctypes.POINTER(ActGeom), _i32, ctypes.POINTER(ActGeom), _vp, _vp]),
    "hfc_spectral_sigma": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "hfc_gan_sums": (ctypes.c_int, [_vp, _i64, _vp, _vp]),
    "hfc_sqdiff_sum": (ctypes.c_int, [_vp, _vp, _i64, _f32, _vp, _vp]),
    "hfc_lpips_layer": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "hfc_gemm_nt": (ctypes.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _i32, _i32, _vp]),
    "hfc_rows_to_act": (ctypes.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _vp, _vp]),
    "hfc_im2col_t": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32,
                                    ctypes.c_char_p, ctypes.c_char_p, _i32, _i64, _vp, _vp]),
    "hfc_permute_wgrad": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, ctypes.c_char_p, ctypes.c_char_p,
                                         _f32, _i32, _vp, _vp]),
    "hfc_col_sums": (ctypes.c_int, [_vp, _i32, _i64, _i32, _f32, _vp, _vp]),
    "hfc_pad_fold": (ctypes.c_int, [_vp, _i32, _i32, _i32, ctypes.POINTER(ActGeom), _i32, _vp, _i32, _vp]),
    "hfc_channelnorm_bwd": (ctypes.c_int, [_vp, _i32, _vp, _i32, _vp, _vp, _i32, _i64, _f32, _i32, _vp, _i32, _vp, _vp, _vp, _vp,
                                          _i32, _i32, _vp]),
    "hfc_instancenorm_ws_bytes": (ctypes.c_int64, [_i32, _i32]),
    "hfc_instancenorm": (ctypes.c_int, [_vp, _i32, ctypes.POINTER(ActGeom), _i32, _vp, _vp, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _i64,
                                       _vp]),
    "hfc_instancenorm_bwd": (ctypes.c_int, [_vp, _i32, _vp, _i32, _vp, _vp, _i32, _i32, _i32, _f32, _i32, _vp, _i32, _vp, _vp, _vp,
                                           _vp, _i32, _i32, _vp, _i64, _vp]),
    "hfc_relu_mask": (ctypes.c_int, [_vp, _i32, _vp, ctypes.POINTER(ActGeom), _f32, _vp, _i32, _vp]),
    "hfc_rows_to_act_geom": (ctypes.c_int, [_vp, _i32, ctypes.POINTER(ActGeom), _i32, _vp, _vp]),
    "hfc_adam_chunk": (ctypes.c_int32, []),
    "hfc_adam_multi": (ctypes.c_int, [_vp, _vp, _i32, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                     ctypes.c_double, _i64, _vp]),
    "hfc_wgrad": (ctypes.c_int, [ctypes.POINTER(WgradDesc), _vp, _vp, _vp, _i32, _vp]),
    "hfc_act_to_bf16": (ctypes.c_int, [_vp, _vp, _i64, _vp]),
    "hfc_disc_input_bwd": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp]),
    "hfc_spectral_bwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp]),
    "hfc_gan_grad": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp]),
    "hfc_latent_likelihood_bwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _f32, _i64, _f32, _i32, _vp, _vp, _vp, _vp]),
    "hfc_hyperlatent_likelihood_bwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _f32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "hfc_lpips_layer_bwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "hfc_conv_forward": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hfc_conv_widenorm_supported": (ctypes.c_int, [ctypes.POINTER(ConvDesc)]),
    "hfc_conv_forward_widenorm": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32,
                                                 _vp, _vp]),
    "hfc_nchw_to_act": (ctypes.c_int, [_vp, ctypes.POINTER(ActGeom), _i32, _i32, _vp, _vp, _f32, _vp, _vp]),
    "hfc_channelnorm": (ctypes.c_int, [_vp, _i32, ctypes.POINTER(ActGeom), _i32, _vp, _vp, _f32, _i32,
                                       _vp, _vp, _vp, _vp, _vp]),
    "hfc_latent_likelihood": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _i32, _vp, _vp, _vp]),
    "hfc_hyperlatent_likelihood": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "hfc_quantize_symbols": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _i32, _f32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "hfc_scale_indices": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _i32, _f32, _i32, _i32, _vp, _vp]),
    "hfc_dequantize_symbols": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "hfc_pmf_to_quantized_cdf_host": (ctypes.c_int, [_vp, _i32, _i32, _vp]),
    "hfc_rans_encode_host": (_i64, [_vp, _vp, _i64, _i64, _vp, _i32, _i32, _vp, _vp, _i32, _vp, _i64]),
    "hfc_rans_decode_host": (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _vp, _i32, _i32, _vp, _vp, _i32, _vp]),
    "hfc_dlmm_likelihood": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "hfc_dlmm_likelihood_bwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _f32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "hfc_lpips_prep": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "hfc_lpips_prep_bwd": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "hfc_maxpool3s2": (ctypes.c_int, [_vp, ctypes.POINTER(ActGeom), _vp, _vp]),
    "hfc_maxpool3s2_bwd": (ctypes.c_int, [_vp, _i32, _vp, ctypes.POINTER(ActGeom), _vp, _i32, _vp]),
    "hfc_lpips_nhwc": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "hfc_lpips_nhwc_bwd": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _i32, _vp]),
    "hfc_ssim_ws_bytes": (ctypes.c_int64, [_i32, _i32, _i32, _i32, _i32, _i32]),
    "hfc_ssim_level": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _f32, _f32, _vp, _vp, _vp, _i64,
                                      _vp]),
    "hfc_ssim_finalize": (ctypes.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _i32, _vp, _i64, _vp, _vp]),
    "hfc_psnr_ws_bytes": (ctypes.c_int64, [_i32, _i64]),
    "hfc_psnr": (ctypes.c_int, [_vp, _vp, _i32, _i64, ctypes.c_double, _vp, _i64, _vp, _vp]),
}


def build(verbose=False):
    """Compile libhfc.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    res = subprocess.run(["make", "-C", CSRC_DIR, "-j4"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise RuntimeError("libhfc build failed")
    return LIB_PATH


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"libhfc.so not found at {LIB_PATH}: build it with `make -C {CSRC_DIR}` or "
            "`python -c 'import __graft_entry__ as g; g.build()'`. There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = ABI mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


class HfcError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        msg = lib.hfc_last_error().decode("utf-8", "replace")
        raise HfcError(f"libhfc {what} failed (status {rc}): {msg}")
