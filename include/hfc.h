/*
 * hfc.h -- C ABI of libhfc (B200 / sm_100a kernels for the HiFIC forward/backward hot path).
 *
 * The reference (Justin-Tan/high-fidelity-generative-compression @ 7d4e9e7) has no FFI of its own:
 * every operator on the hot path is an eager torch call issued from its nn.Module classes.  The
 * entry points below are therefore cut at exactly those call sites -- one entry point per torch
 * operator group the reference issues -- so a maintainer can bind them from the reference modules
 * with ctypes (see INTEGRATION.md).  Each declaration cites the reference lines it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types; all pointers are DEVICE pointers unless the
 *     name ends in _host;
 *   - every call enqueues work on the caller's `stream` (a cudaStream_t passed as void*) and
 *     returns without synchronising;
 *   - returns 0 on success, a negative hfc_status otherwise; never throws; hfc_last_error()
 *     gives a thread-local message;
 *   - the library never allocates device memory: the caller owns inputs, outputs and workspaces;
 *   - there is NO CPU fallback: on a machine without an sm_100 GPU the compute calls return
 *     HFC_ERR_NO_DEVICE.
 *
 * Internal activation format ("act buffer"): NHWC, 16-bit (fp16, or bf16 hi/lo planes in the
 * split-precision mode), channels padded to `cpad` (multiple of 8; multiples of 64 for conv
 * inputs), with an optional materialised spatial border (pt, pl, pb, pr) that the PRODUCING
 * kernel fills by reflection so that the consuming convolution's ReflectionPad2d is free.
 */
#ifndef HFC_H_
#define HFC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HFC_ABI_VERSION 1

typedef enum hfc_status {
  HFC_OK = 0,
  HFC_ERR_INVALID = -1,     /* bad descriptor / unsupported combination */
  HFC_ERR_NO_DEVICE = -2,   /* no sm_100 device or driver entry point missing */
  HFC_ERR_LAUNCH = -3,      /* CUDA launch / runtime error (message has the CUDA string) */
  HFC_ERR_UNSUPPORTED = -4  /* valid request that this build does not implement */
} hfc_status;

enum { HFC_PAD_ZERO = 0, HFC_PAD_REFLECT = 1 };
enum { HFC_ACT_NONE = 0, HFC_ACT_RELU = 1, HFC_ACT_LEAKY02 = 2 };
enum { HFC_OUT_NHWC_F16 = 0, HFC_OUT_NHWC_F32 = 1, HFC_OUT_NCHW_F32 = 2 };
enum { HFC_PREC_F16 = 0, HFC_PREC_BF16X3 = 1 };

/* NHWC 16-bit activation buffer geometry (see "Internal activation format"). */
typedef struct hfc_act_geom {
  int32_t n, h, w;          /* logical batch / height / width (without border) */
  int32_t c, cpad;          /* real and padded channel count */
  int32_t pt, pl, pb, pr;   /* materialised border rows/cols (top, left, bottom, right) */
} hfc_act_geom;

/*
 * One convolution / transposed convolution as issued by the reference:
 *   F.conv2d            : src/network/encoder.py:56-101, generator.py:33-44,98-103,139-142,
 *                         hyper.py:52-63, discriminator.py:66-86
 *   F.conv_transpose2d  : src/network/generator.py:115-137, hyper.py:83-97
 * fused (optionally) with what follows it in the reference module:
 *   bias, ChannelNorm2D (src/normalisation/channel.py:48-59), ReLU / LeakyReLU(0.2),
 *   and the ReflectionPad2d of the NEXT layer (materialised into the output border).
 */
typedef struct hfc_conv_desc {
  hfc_act_geom in;          /* input act buffer */
  int32_t kh, kw;           /* filter size */
  int32_t stride;           /* 1 or 2 */
  int32_t transposed;       /* 0: conv2d, 1: conv_transpose2d (output_padding = stride-1) */
  int32_t pad_mode;         /* HFC_PAD_ZERO | HFC_PAD_REFLECT (reflect needs in.p* >= pad_*) */
  int32_t pad_t, pad_l, pad_b, pad_r; /* logical padding; for transposed: `padding` arg in pad_t/pad_l */
  int32_t cout;             /* real output channels */
  int32_t window;           /* 1: 'window' packing for tiny cin (cin<=8, cpad==8, kw<=8): one
                               K block covers a whole filter row (kw x cin) */
  /* output */
  int32_t out_mode;         /* HFC_OUT_* */
  hfc_act_geom out;         /* NHWC_F16: full geometry; NHWC_F32: cpad = row pitch in floats,
                               borders ignored; NCHW_F32: plain (n, cout, h, w) */
  int32_t out_reflect;      /* fill out border by reflection (NHWC_F16 only) */
  int32_t act;              /* HFC_ACT_* applied after bias (and after the norm when fused) */
  int32_t norm;             /* 1: fuse ChannelNorm2D (needs cout <= 256) */
  float eps;                /* ChannelNorm eps (reference: 1e-3) */
  int32_t block_n;          /* 0 = auto; else N tile (multiple of 16, <= 256) */
  int32_t precision;        /* HFC_PREC_* */
  int32_t cluster_m;        /* 0 = auto; else 1 or 2: CTAs per cluster along M tiles (share the weight tile) */
  int32_t cluster_n;        /* 0 = auto; else 1 or 2: CTAs per cluster along N tiles (share the pixel tile) */
  int32_t wide;             /* tiny-cout convs on big maps (the 7x7 60->3 head): 0 = auto (tap-in-N), 1 = force the
                               row-resident 'wide' mode (halo row + resident weights, filter columns by descriptor
                               shift), 2 = forbid both, 3 = force 'tap-in-N' (GEMM columns = (filter column, cout),
                               filter columns summed with a pixel shift in the epilogue) */
  int32_t a_bf16, b_bf16;   /* operand formats: 0 = fp16, 1 = bf16 (activation operand / weight operand); the backward
                               pass feeds bf16 gradients against fp16 activations / weights */
  int32_t dgrad;            /* 1: pack the weights for the data gradient of a stride-1 conv2d: W'[ci][co][r][s] =
                               W[co][ci][kh-1-r][kw-1-s] (cout of this descriptor = cin of the forward conv) */
  int32_t pair;             /* 0 = auto, 1 = force, 2 = forbid CTA pairs (cta_group::2 UMMA, M = 256 over two SMs;
                               needs cluster_m == 2) */
} hfc_conv_desc;

typedef struct hfc_conv_info {
  size_t packed_weight_bytes;   /* size of the packed weight buffer hfc_conv_pack_weights fills */
  int32_t out_h, out_w;         /* logical output dims */
  int32_t phases;               /* kernel launches per forward (4 for stride-2 transposed) */
  int32_t block_n, n_tiles, m_tiles, stages, k_total;
  int32_t cluster_m, cluster_n; /* cluster shape the launch will use (TMA multicast) */
  int32_t wide;                 /* 1 if the row-resident 'wide' mode is used */
  int32_t pair;                 /* 1 if CTA pairs (cta_group::2) are used */
  int32_t tapn;                 /* 1 if the tap-in-N mode is used */
  int32_t nsub;                 /* N tiles per work item (2: CTA pairs with one N tile in each TMEM half) */
  double flops;                 /* algorithmic 2*MACs of the layer (real channels) */
} hfc_conv_info;

/* library / device */
int hfc_abi_version(void);
const char* hfc_last_error(void);
int hfc_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* number of kernels this library has launched in the calling process (bench.py: gpu_launches) */
unsigned long long hfc_launch_count(void);

/* convolution */
int hfc_conv_query(const hfc_conv_desc* d, hfc_conv_info* info);
/* w: fp32 (cout, cin, kh, kw) for conv2d, (cin, cout, kh, kw) for conv_transpose2d (torch layout) */
int hfc_conv_pack_weights(const hfc_conv_desc* d, const float* w, void* packed, void* stream);
/* same, with every weight multiplied by *scale (a DEVICE scalar), e.g. 1/sigma of spectral normalisation
 * (torch.nn.utils.spectral_norm divides weight_orig by sigma, src/network/discriminator.py:46-62) */
int hfc_conv_pack_weights_scaled(const hfc_conv_desc* d, const float* w, const float* scale, void* packed,
                                 void* stream);
/* in: act buffer (d->in); packed: from hfc_conv_pack_weights; bias/gamma/beta: fp32 [cout] or NULL;
 * out: buffer of d->out_mode/d->out */
int hfc_conv_forward(const hfc_conv_desc* d, const void* in, const void* packed, const float* bias,
                     const float* gamma, const float* beta, void* out, void* stream);
/*
 * Convolution fused with a ChannelNorm2D over a channel row that does NOT fit one accumulator tile (768 < cout <= 1024:
 * the Generator's 960-channel residual trunk, src/network/generator.py:33-44): the row of a pixel lives in the four TMEM
 * halves of two CTA pairs of a 4-CTA cluster, which exchange per-pixel (mean, M2) through distributed shared memory;
 * y = act(gamma * (x - mean) * rsqrt(var_unbiased + eps) + beta) [+ res1] [+ res2] is written as fp32 rows (out_f32,
 * pitch ld_f32; optional) and into the bordered NHWC fp16 buffer described by d->out (out_act; optional) -- i.e.
 * hfc_conv_forward(NHWC_F32) + hfc_channelnorm in one launch.  d: a stride-1 / stride-2 conv2d descriptor with norm = 1,
 * out_mode = HFC_OUT_NHWC_F16, cout % 16 == 0; res1 / res2: fp32 rows of pitch ld_res (may be NULL).
 * Returns HFC_ERR_UNSUPPORTED for geometries whose pixel tiles do not pair up (callers then use the two-launch path).
 */
/* HFC_OK if hfc_conv_forward_widenorm can run this descriptor (host-only check, works without a GPU) */
int hfc_conv_widenorm_supported(const hfc_conv_desc* d);
int hfc_conv_forward_widenorm(const hfc_conv_desc* d, const void* in, const void* packed, const float* bias,
                              const float* gamma, const float* beta, const float* res1, const float* res2,
                              int32_t ld_res, float* out_f32, int32_t ld_f32, void* out_act, void* stream);

/*
 * Layout conversion at module boundaries (the reference modules exchange NCHW fp32):
 * x (n, c, h, w) fp32 -> act buffer `g` (border by reflection or zeros), optionally applying
 * ChannelNorm2D first (Generator.conv_block_init[0], src/network/generator.py:98-103).
 */
int hfc_nchw_to_act(const float* x, const hfc_act_geom* g, int32_t reflect, int32_t norm,
                    const float* gamma, const float* beta, float eps, void* out, void* stream);

/*
 * Stand-alone ChannelNorm2D (src/normalisation/channel.py:48-59) for channel counts that do not
 * fit one accumulator tile (480, 960): x = raw conv output, NHWC fp32 rows of pitch `ld`;
 * y = act(gamma * (x - mean) * rsqrt(var_unbiased + eps) + beta) [+ res1] [+ res2];
 * writes y as fp32 rows (out_f32, optional) and as act buffer `g` (out_act, optional).
 * res1/res2 implement ResidualBlock's `torch.add(res, identity_map)` (generator.py:44) and
 * Generator's `x += head` (generator.py:161).
 */
int hfc_channelnorm(const float* x, int32_t ld, const hfc_act_geom* g, int32_t reflect,
                    const float* gamma, const float* beta, float eps, int32_t act,
                    const float* res1, const float* res2, float* out_f32, void* out_act,
                    void* stream);

/*
 * Hyperprior likelihoods (src/hyperprior.py:57-139, 277-330; src/helpers/maths.py:87-109;
 * src/compression/hyperprior_model.py:305-384).  All tensors NCHW fp32.
 *
 * hfc_latent_likelihood: one pass over (y, mean, scale_raw[, noise]):
 *   scale = max(scale_raw, scale_lower_bound)                        (LowerBoundToward)
 *   noisy  = y + noise ; p_n = Phi((.5-|noisy-mean|)/scale) - Phi(-(.5+|noisy-mean|)/scale)
 *   quant  = floor(y-mean+.5)+mean ; p_q likewise ;  p = max(p, 1e-9)
 *   sums[0] += sum log(p_n + 1e-9) ; sums[1] += sum log(p_q + 1e-9)   (natural log, fp64 accum)
 *   decoded = quant (the straight-through value, hyperprior.py:108-122)
 * likelihood_type: 0 gaussian (erfc), 1 logistic (sigmoid).  noise may be NULL (=> no noisy term).
 * `sums` (2 doubles) must be zeroed by the caller.
 */
int hfc_latent_likelihood(const float* y, const float* mean, const float* scale_raw,
                          const float* noise, int64_t count, float scale_lower_bound,
                          int32_t likelihood_type, float* decoded, double* sums, void* stream);
/*
 * hfc_hyperlatent_likelihood: factorized density (4-layer monotone MLP per channel) evaluated at
 * z+noise and at round(z):  z (n, c, h, w); params packed per channel as 44 floats:
 *   softplus(H0)[3], b0[3], tanh(a0)[3], softplus(H1)[3x3 row-major], b1[3], tanh(a1)[3],
 *   softplus(H2)[3x3], b2[3], tanh(a2)[3], softplus(H3)[3], b3[1], tanh(a3)[1]
 *   (each channel's block padded to 64 floats)
 * outputs: z_noisy, z_quant (either may be NULL), sums[0] (noisy) and sums[1] (quantised) as above.
 */
int hfc_hyperlatent_likelihood(const float* z, const float* noise, const float* params64,
                               int32_t n, int32_t c, int32_t hw, float* z_noisy, float* z_quant,
                               double* sums, void* stream);

/*
 * Discriminator input (src/network/discriminator.py:75-79): torch.cat((x, Upsample(scale, 'nearest')(ctx)), 1)
 * written straight into the bordered NHWC act buffer conv1 reads.  x: (n, x_channels, h, w) fp32 NCHW;
 * ctx_act: border-less act buffer `ctx` (n, h/scale, w/scale, c) from the context conv.
 */
int hfc_disc_input(const float* x, int32_t x_channels, const void* ctx_act, const hfc_act_geom* ctx,
                   int32_t scale, const hfc_act_geom* out_geom, void* out, void* stream);

/*
 * Spectral norm of a (rows x cols) row-major weight matrix as torch.nn.utils.spectral_norm computes it:
 * power_iteration != 0 (training): v = normalize(W^T u), u = normalize(W v) (u, v updated in place),
 * sigma = u.(W v); power_iteration == 0 (eval): sigma = u.(W v) from the stored u, v.
 * workspace: rows + cols floats.  sigma / inv_sigma: device scalars (inv_sigma may be NULL).
 */
int hfc_spectral_sigma(const float* w, int32_t rows, int32_t cols, float* u, float* v, int32_t power_iteration,
                       float* workspace, float* sigma, float* inv_sigma, void* stream);

/*
 * GAN loss sums (src/loss/losses.py:30-41): logits = [real | generated] halves of half_count elements;
 * sums5 (caller-zeroed doubles): sum BCE(real,1), sum BCE(gen,0), sum BCE(gen,1), sum sigmoid(real),
 * sum sigmoid(gen).
 */
int hfc_gan_sums(const float* logits, int64_t half_count, double* sums5, void* stream);

/* Distortion loss sum (src/model.py:190-194): *sum += sum((scale*a - scale*b)^2); caller zeroes *sum. */
int hfc_sqdiff_sum(const float* a, const float* b, int64_t count, float scale, double* sum, void* stream);

/*
 * LPIPS feature loss of one trunk layer (src/loss/perceptual_similarity/networks_basic.py:61-89,
 * perceptual_loss.py:42-46): f0, f1 (n, c, h*w) fp32 trunk features of the two images, lin_w (c) the
 * non-negative 1x1 'lin' weights; out_per_image[i] += mean_hw sum_c w_c (f0/|f0| - f1/|f1|)^2.
 */
int hfc_lpips_layer(const float* f0, const float* f1, const float* lin_w, int32_t n, int32_t c, int32_t hw,
                    float* out_per_image, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Backward pass building blocks (autograd of F.conv2d / F.conv_transpose2d, train.py:49-59).
 *   data gradient   : hfc_conv_forward on the gradient tensor with the transposed role of the weights
 *                     (stride-1 conv: desc.dgrad = 1; stride-2 conv: a transposed conv; transposed conv: a conv)
 *   weight gradient : one GEMM  dW[c1][(tap, c2)] = A1T[c1][pixels] * COLT[(tap, c2)][pixels]^T
 * Gradients travel between layers as fp32 rows [pixels][channels]; GEMM operands made of them are bf16.
 * --------------------------------------------------------------------------------------------------------- */
/* C[m][n] (fp32, row pitch ldc, overwritten) = A[m][k] * B[n][k]^T; A, B: K-major 16-bit (fp16 or bf16), k % 64 == 0.
 * k_splits: 0 = auto, else number of K partitions accumulated with fp32 atomics (C is zeroed first). */
int hfc_gemm_nt(const void* a, int32_t a_bf16, const void* b, int32_t b_bf16, int32_t m, int32_t n, int32_t k,
                float* c, int32_t ldc, int32_t k_splits, void* stream);
/* fp32 rows [npix][ld] -> border-less 16-bit act buffer [npix][cpad] (bf16 if to_bf16 else fp16), padding = 0 */
int hfc_rows_to_act(const float* rows, int32_t ld, int64_t npix, int32_t c, int32_t cpad, int32_t to_bf16, void* out,
                    void* stream);
/* same, into the INTERIOR of the bordered buffer described by g (the border is not written: zero it once) */
int hfc_rows_to_act_geom(const float* rows, int32_t ld, const hfc_act_geom* g, int32_t to_bf16, void* out, void* stream);
/* transposed im2col (see csrc/backward.cu): out[(tap*c_rows + ch)][p], p over the (n, gh, gw) pixel grid, source
 * coordinate (g*stride + d[tap] + o0) in a physical buffer of n x hp x wp pixels with cpad channels (pitch, for fp32
 * rows), zero outside; src_f32: 0 = 16-bit source copied verbatim, 1 = fp32 rows converted to bf16 (3: to fp16), 2 = fp16 act
 * buffer converted to bf16 (the backward GEMMs run bf16 x bf16).
 * dh_host / dw_host are HOST arrays of ntaps offsets. */
int hfc_im2col_t(const void* src, int32_t src_f32, int32_t n, int32_t hp, int32_t wp, int32_t cpad, int32_t c_src,
                 int32_t gh, int32_t gw, int32_t stride, int32_t oh0, int32_t ow0, int32_t ntaps,
                 const int8_t* dh_host, const int8_t* dw_host, int32_t c_rows, int64_t p_pad, void* out, void* stream);
/* GEMM result C[m][(tap, c2)] -> dW[m][c2][ky][kx] (torch layout) * scale (+= if accumulate) */
int hfc_permute_wgrad(const float* c, int32_t ldc, int32_t m, int32_t c2, int32_t c2_rows, int32_t kh, int32_t kw,
                      int32_t ntaps, const int8_t* ky_host, const int8_t* kx_host, float scale, int32_t accumulate,
                      float* dw, void* stream);
/* torch.optim.Adam step (amsgrad = False) over a list of fp32 tensors in one launch (train.py:287-300, 54-59).
 * table_dev: 5 x int64 per tensor {param ptr, grad ptr, exp_avg ptr, exp_avg_sq ptr, numel};
 * blockmap_dev: 2 x int32 per block {tensor index, chunk index}, one block per hfc_adam_chunk() elements;
 * step: the 1-based step count used for the bias corrections. */
int32_t hfc_adam_chunk(void);
int hfc_adam_multi(const int64_t* table_dev, const int32_t* blockmap_dev, int32_t n_blocks, double lr, double beta1,
                   double beta2, double eps, double weight_decay, int64_t step, void* stream);
/* Implicit weight gradient (autograd of F.conv2d / F.conv_transpose2d w.r.t. the weight, train.py:49-59):
 *   c[m][tap * c2_rows + j] = sum over the pixels p of `plain`  plain[p][m] * shifted[p * stride + tap][j]
 * with c2_rows = round_up(shifted.c, 64).  Both operands are NHWC 16-bit activation buffers (same format: fp16 or
 * bf16) with channel pitches that are multiples of 64; tap offsets are relative to the interior origin of `shifted`
 * (negative / overhanging positions read its materialised border or zeros outside the buffer).
 * conv2d: plain = dL/dy (m = cout), shifted = layer input, tap = (ky - pad_t, kx - pad_l);
 * conv_transpose2d: plain = layer input (m = cin), shifted = dL/dy, tap = (ky - pad, kx - pad). */
typedef struct hfc_wgrad_desc {
  hfc_act_geom plain;
  hfc_act_geom shifted;
  int32_t ntaps;
  int32_t stride;      /* sampling stride in `shifted` (1 or 2) */
  int32_t bf16;        /* operand format: 0 fp16, 1 bf16 */
  int32_t k_splits;    /* 0 = auto; > 1 splits the pixels across CTAs (fp32 atomics into c, which is zeroed first) */
  int32_t pair;        /* 0 = auto (CTA pairs, cta_group::2, when both operands are wide enough), 2 = never */
  int32_t window;      /* 1: `shifted` has an 8-channel pitch; column j of a tap = (pixel offset j / 8, channel j % 8) of the
                        * 8-pixel window that starts at the tap position (taps then enumerate filter ROWS only) */
  int8_t tap_dh[64];
  int8_t tap_dw[64];
} hfc_wgrad_desc;
int hfc_wgrad(const hfc_wgrad_desc* d, const void* plain, const void* shifted, float* c, int32_t ldc, void* stream);
/* fp16 -> bf16 copy of an activation buffer (count 16-bit elements, multiple of 8) */
int hfc_act_to_bf16(const void* src_f16, void* dst_bf16, int64_t count, void* stream);
/* out[c] += scale * sum over rows of rows[.][c]   (bias gradient) */
int hfc_col_sums(const float* rows, int32_t ld, int64_t npix, int32_t c, float scale, float* out, void* stream);
/* adjoint of the materialised padding: gradient over the padded domain (fp32 rows of an n x hq x wq grid, pitch
 * ld_in) -> gradient of the un-padded (n, h, w, c) tensor (fp32 rows, pitch ld_out); reflect: mirrored positions add */
int hfc_pad_fold(const float* dxp, int32_t ld_in, int32_t hq, int32_t wq, const hfc_act_geom* g, int32_t reflect,
                 float* dx, int32_t ld_out, void* stream);

/* ChannelNorm2D (+ReLU) backward: z = saved pre-norm rows, g = gradient w.r.t. the block output (both fp32 rows);
 * writes dz (fp32 rows) and ACCUMULATES dgamma / dbeta (caller zeroes them) and, when dbias != NULL, the column sums
 * of dz (= gradient of the bias of the convolution in front of the norm).  dz (fp32 rows) and / or dz_act (16-bit:
 * bf16 if act_bf16 else fp16; border-less NHWC with pitch act_cpad, channel padding zeroed: the operand of the backward
 * GEMMs) receive the result; either may be NULL.  act: HFC_ACT_NONE | HFC_ACT_RELU. */
int hfc_channelnorm_bwd(const float* z, int32_t ld_z, const float* g, int32_t ld_g, const float* gamma,
                        const float* beta, int32_t c, int64_t npix, float eps, int32_t act, float* dz, int32_t ld_dz,
                        float* dgamma, float* dbeta, float* dbias, void* dz_act, int32_t act_cpad, int32_t act_bf16,
                        void* stream);
/*
 * InstanceNorm2d variant of the inter-layer normalisation (use_channel_norm = False: src/normalisation/instance.py:7-15 ->
 * torch.nn.InstanceNorm2d(affine=True, track_running_stats=False), selected in src/network/encoder.py:41-44 and
 * src/network/generator.py:21-24, 81-84).  Same contract as hfc_channelnorm, but the statistics are per (image, channel)
 * over the h*w pixels (biased variance):  y = act(gamma * (x - mean_nc) * rsqrt(var_nc + eps) + beta) [+ res1] [+ res2],
 * written as fp32 rows (out_f32, pitch c, optional) and as the bordered act buffer `g` (out_act, optional).
 * ws: device scratch of at least hfc_instancenorm_ws_bytes(n, c) bytes (8-byte aligned; contents are overwritten).
 */
int64_t hfc_instancenorm_ws_bytes(int32_t n, int32_t c);
int hfc_instancenorm(const float* x, int32_t ld, const hfc_act_geom* g, int32_t reflect, const float* gamma,
                     const float* beta, float eps, int32_t act, const float* res1, const float* res2, float* out_f32,
                     void* out_act, void* ws, int64_t ws_bytes, void* stream);
/* Autograd of hfc_instancenorm (torch.nn.InstanceNorm2d + ReLU as encoder.py:56-61 / generator.py:33-44 chain them):
 * z [n*hw][ld_z] = the saved norm input, g [n*hw][ld_g] = the gradient of the norm output.  dz as fp32 rows and / or
 * as the 16-bit operand of the backward GEMMs (dz_act, pitch act_cpad, bf16 if act_bf16 else saturating fp16); dgamma /
 * dbeta / dbias (optional; = column sums of dz) are ACCUMULATED into the caller's (zeroed) buffers. */
int hfc_instancenorm_bwd(const float* z, int32_t ld_z, const float* g, int32_t ld_g, const float* gamma, const float* beta,
                         int32_t c, int32_t n, int32_t hw, float eps, int32_t act, float* dz, int32_t ld_dz, float* dgamma,
                         float* dbeta, float* dbias, void* dz_act, int32_t act_cpad, int32_t act_bf16, void* ws,
                         int64_t ws_bytes, void* stream);
/* out = g * (y > 0 ? 1 : slope): backward of the fused bias + ReLU (slope 0) / LeakyReLU (slope 0.2) epilogue; y_act
 * is that layer's (bordered) NHWC fp16 output */
int hfc_relu_mask(const float* g, int32_t ld_g, const void* y_act, const hfc_act_geom* geom, float slope, float* out,
                  int32_t ld_out, void* stream);
/* adjoint of hfc_disc_input (autograd of torch.cat + nn.Upsample(nearest), src/network/discriminator.py:75-79):
 * g = gradient rows [n*h*w][ld_g] of the (x_channels + ctx_channels)-channel discriminator input; dx (NCHW fp32,
 * may be NULL) receives the image part, dctx rows [n*(h/scale)*(w/scale)][ld_ctx] the scale x scale block sums. */
int hfc_disc_input_bwd(const float* g, int32_t ld_g, int32_t n, int32_t h, int32_t w, int32_t x_channels,
                       int32_t ctx_channels, int32_t scale, float* dx, float* dctx, int32_t ld_ctx, void* stream);
/* backward of torch.nn.utils.spectral_norm's W = W_orig / sigma (discriminator.py:46-62; u, v are constants):
 * dw_orig (+)= (dw - <dw, W> u v^T) * inv_sigma.  workspace1: one float of scratch. */
int hfc_spectral_bwd(const float* dw, const float* w_orig, const float* u, const float* v, const float* inv_sigma,
                     int32_t rows, int32_t cols, float* workspace1, int32_t accumulate, float* dw_orig, void* stream);
/* d loss / d logits of the non-saturating GAN losses (src/loss/losses.py:30-41) for logits = [real (half_count),
 * gen (half_count)]; mode 0 = generator loss, 1 = discriminator loss; upstream = device scalar d L / d loss or NULL */
int hfc_gan_grad(const float* logits, int64_t half_count, int32_t mode, const float* upstream, float* dlogits,
                 void* stream);
/* backward of hfc_latent_likelihood's noisy term: L = (*g_nbpp) * coef * sum ln(p_noisy + 1e-9); dyhat = upstream
 * gradient of the straight-through latents (may be NULL).  All NCHW fp32. */
int hfc_latent_likelihood_bwd(const float* y, const float* mean, const float* scale_raw, const float* noise,
                              const float* dyhat, const float* g_nbpp, float coef, int64_t count,
                              float scale_lower_bound, int32_t likelihood_type, float* dy, float* dmean, float* dscale,
                              void* stream);
/* backward of hfc_hyperlatent_likelihood's noisy term w.r.t. the noisy hyper-latents (dz = dz_in + ...) and the
 * PACKED density parameters (dparams64, overwritten, same (c, 64) layout) */
int hfc_hyperlatent_likelihood_bwd(const float* z_noisy, const float* dz_in, const float* params64,
                                   const float* g_nbpp, float coef, int32_t n, int32_t c, int32_t hw, float* dz,
                                   float* dparams64, void* stream);
/* gradient of hfc_lpips_layer w.r.t. f1 (the reconstruction's features): df1 = upstream[image] * d(mean dist)/d f1 */
int hfc_lpips_layer_bwd(const float* f0, const float* f1, const float* lin_w, const float* upstream, int32_t n,
                        int32_t c, int32_t hw, float* df1, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Compress / decompress path (compress.py, src/model.py:262-344, src/hyperprior.py:195-274): the GPU half
 * (symbols, table indices, Shannon bits, dequantisation) and the HOST half (table quantisation, the rANS coder
 * -- "the sequential ANS entropy coder stays on the host", BASELINE north_star).  *_host functions take HOST
 * pointers, do not touch the GPU and work without one.
 * --------------------------------------------------------------------------------------------------------- */
/* layout of the symbol arrays the vectorised coder walks, [steps][lanes] (entropy_coding.py:298-316 with
 * PATCH_SIZE (1, 1)): HFC_SYM_BATCH_STEPS: steps = n, lanes = (c, h, w) (plain NCHW, the reference's batch > 1 case);
 * HFC_SYM_PIXEL_STEPS: steps = (n, h, w), lanes = c (the reference's batch == 1 case, n must be 1 there). */
enum { HFC_SYM_BATCH_STEPS = 0, HFC_SYM_PIXEL_STEPS = 1 };
/*
 * Encoder side of PriorEntropyModel.compress (src/compression/prior_model.py:148-198) fused with
 * _estimate_compression_bits (:122-146) -- and of HyperpriorEntropyModel.compress (hyperprior_model.py:141-197)
 * when mean == NULL and scale_raw == NULL:
 *   symbols = (int32) floor(x + 0.5 - mean)
 *   indices = 63 - #{ s in scale_table[0..n_scales-2] : max(scale_raw, scale_lower_bound) <= s }   (compute_indices)
 *             (scale_raw == NULL: indices = channel)
 *   dequant = symbols + mean   (what the decoder reconstructs; optional, NCHW fp32)
 *   *bits_sum += sum ln(max(p, 1e-9) + 1e-9), p = conditional likelihood of the quantised value (optional, fp64,
 *               caller-zeroed; only with scale_raw; natural log: divide by -ln 2 for bits)
 * x / mean / scale_raw / dequant: NCHW fp32; symbols / indices: int32 in `layout` order.
 * table_sorted: 1 if scale_table is non-decreasing (the caller checks; the reference's log-spaced table is): the
 * index is then found by binary search -- same integers as the reference's compare loop -- else by the linear count.
 */
int hfc_quantize_symbols(const float* x, const float* mean, const float* scale_raw, int32_t n, int32_t c, int32_t hw,
                         const float* scale_table, int32_t n_scales, float scale_lower_bound, int32_t likelihood_type,
                         int32_t layout, int32_t table_sorted, int32_t* symbols, int32_t* indices, float* dequant,
                         double* bits_sum, void* stream);
/* Decoder side (prior_model.py:201-246, entropy_models.py:65-73): symbols (int32, `layout` order) -> NCHW fp32
 * out = symbols + mean (mean may be NULL). */
int hfc_dequantize_symbols(const int32_t* symbols, const float* mean, int32_t n, int32_t c, int32_t hw, int32_t layout,
                           float* out, void* stream);
/* Decoder side of compute_indices alone (prior_model.py:148-156): indices in `layout` order from NCHW scale_raw. */
int hfc_scale_indices(const float* scale_raw, int32_t n, int32_t c, int32_t hw, const float* scale_table,
                      int32_t n_scales, float scale_lower_bound, int32_t layout, int32_t table_sorted, int32_t* indices,
                      void* stream);

/* maths.pmf_to_quantized_cdf (src/helpers/maths.py:5-73): n float32 probabilities -> n + 1 integers, cdf[0] = 0,
 * cdf[n] = 2^precision, every symbol keeps a non-zero frequency. */
int hfc_pmf_to_quantized_cdf_host(const float* pmf_host, int32_t n, int32_t precision, int32_t* cdf_host);
/*
 * The reference's vectorised indexed rANS coder (src/compression/entropy_coding.py:251-476, 555-676 over
 * src/compression/ans.py): one 64-bit state per lane, `steps` symbols per lane, symbols / indices int32 [steps][lanes];
 * cdf (cdf_rows x cdf_cols) int32 row-major with cdf_length / cdf_offset per row; symbols outside
 * [offset, offset + length - 2) are escaped with 4-bit codes exactly as the reference does.
 * encode: returns the number of 32-bit words written to out_host (the flat message of ans.flatten), or, with
 * out_host == NULL, the number of words needed; negative hfc_status on error.
 */
int64_t hfc_rans_encode_host(const int32_t* symbols_host, const int32_t* indices_host, int64_t steps, int64_t lanes,
                             const int32_t* cdf_host, int32_t cdf_rows, int32_t cdf_cols,
                             const int32_t* cdf_length_host, const int32_t* cdf_offset_host, int32_t precision,
                             uint32_t* out_host, int64_t out_capacity);
int hfc_rans_decode_host(const uint32_t* encoded_host, int64_t n_words, const int32_t* indices_host, int64_t steps,
                         int64_t lanes, const int32_t* cdf_host, int32_t cdf_rows, int32_t cdf_cols,
                         const int32_t* cdf_length_host, const int32_t* cdf_offset_host, int32_t precision,
                         int32_t* symbols_host);

/* ---------------------------------------------------------------------------------------------------------
 * LPIPS (AlexNet) trunk in the internal activation format (SURVEY.md 8f-1): the non-convolution pieces of
 * src/loss/perceptual_similarity/{perceptual_loss.py:26-46, networks_basic.py:61-98, pretrained_networks.py:56-94}.
 * The trunk's five convolutions are hfc_conv_forward launches (the 11x11 stride-4 head as a 3x3 conv over the 4x4
 * space-to-depth image that hfc_lpips_prep writes); the frozen trunk needs data gradients only.
 * --------------------------------------------------------------------------------------------------------- */
/* target, pred: (n, 3, h, w) fp32 NCHW -> out_act (2n, hs, ws, 64) fp16 border-less, images [0, n) = target, [n, 2n) =
 * pred; channel (dy * 4 + dx) * 3 + c of s2d pixel (I, J) = ((normalize ? 2x - 1 : x) - shift3[c]) / scale3[c] at image
 * position (4I + dy - 2, 4J + dx - 2), zero outside the image; channels 48..63 zero.  hs = ((h + 4 - 11) / 4 + 1) + 2. */
int hfc_lpips_prep(const float* target, const float* pred, int32_t n, int32_t h, int32_t w, int32_t hs, int32_t ws,
                   int32_t normalize, const float* shift3, const float* scale3, void* out_act, void* stream);
/* adjoint for the pred half: g_rows fp32 [n * hs * ws][ld >= 48] -> dpred (n, 3, h, w) */
int hfc_lpips_prep_bwd(const float* g_rows, int32_t ld, int32_t n, int32_t h, int32_t w, int32_t hs, int32_t ws,
                       int32_t normalize, const float* scale3, float* dpred, void* stream);
/* nn.MaxPool2d(kernel_size=3, stride=2) on a border-less NHWC fp16 buffer g -> (n, (h-3)/2+1, (w-3)/2+1, cpad) */
int hfc_maxpool3s2(const void* in_act, const hfc_act_geom* g, void* out_act, void* stream);
/* its adjoint: g_out_rows fp32 [n * oh * ow][ld_out] -> ADDED into g_in_rows fp32 [n * h * w][ld_in] (caller zeroes) at
 * the first maximum of every window (ATen semantics); in_act / g describe the pooled layer's input */
int hfc_maxpool3s2_bwd(const float* g_out_rows, int32_t ld_out, const void* in_act, const hfc_act_geom* g,
                       float* g_in_rows, int32_t ld_in, void* stream);
/* hfc_lpips_layer on one NHWC fp16 feature buffer (2n, hw, cpad) holding target [0, n) and reconstruction [n, 2n):
 * out_per_image[i] += mean_hw sum_c lin_w[c] (f0/|f0| - f1/|f1|)^2 */
int hfc_lpips_nhwc(const void* feat_act, int32_t n, int32_t hw, int32_t c, int32_t cpad, const float* lin_w,
                   float* out_per_image, void* stream);
/* gradient w.r.t. the PRE-ReLU value of the reconstruction's features: g_out_rows[p][k] = (f1 > 0) *
 * (upstream[img] * d dist / d f1 + g_in_rows[p][k]) ; g_in_rows (the gradient arriving from deeper layers) may be NULL */
int hfc_lpips_nhwc_bwd(const void* feat_act, int32_t n, int32_t hw, int32_t c, int32_t cpad, const float* lin_w,
                       const float* upstream, const float* g_in_rows, int32_t ld_g, float* g_out_rows, int32_t ld_out,
                       void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Discretised mixture likelihood of the latents (`-LMM`; HyperpriorDLMM, src/hyperprior.py:340-458,
 * unpack_likelihood_params src/network/hyper.py:19-35).  x, noise, decoded: (n, c, hw) fp32; dlmm_params: the
 * synthesis network's output (n, 3*c*k, hw), plane (s*c + ch)*k + j with s = 0 mixture logits, 1 means, 2 log-scales.
 *   L(v) = logsumexp_j [log_softmax(logit)_j + log max(Phi(e^{-ls_j}(.5-|v-mu_j|)) - Phi(e^{-ls_j}(-.5-|v-mu_j|)), 1e-9)],
 *   ls_j = max(log-scale_j, -3);  sums[0] += sum L(x + noise) (skipped when noise == NULL), sums[1] += sum L(floor(x+.5));
 *   decoded = straight_through ? x + (floor(x+.5) - x) : floor(x+.5)   (hyperprior.py:443-446).
 * --------------------------------------------------------------------------------------------------------- */
int hfc_dlmm_likelihood(const float* x, const float* noise, const float* dlmm_params, int32_t n, int32_t c, int32_t k,
                        int32_t hw, int32_t likelihood_type, int32_t straight_through, float* decoded, double* sums,
                        void* stream);
/* gradient of (*g_nbpp) * coef * sum L(x + noise) w.r.t. x (dx = d_decoded + ...; d_decoded may be NULL) and w.r.t.
 * dlmm_params (dparams, same layout, overwritten), with both LowerBoundToward gates (pmf >= 1e-9, log-scale >= -3) */
int hfc_dlmm_likelihood_bwd(const float* x, const float* noise, const float* dlmm_params, const float* d_decoded,
                            const float* g_nbpp, float coef, int32_t n, int32_t c, int32_t k, int32_t hw,
                            int32_t likelihood_type, float* dx, float* dparams, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Image-quality metrics of the evaluation loop (compress.py --metrics), src/helpers/metrics.py.  x, y: fp32 NCHW
 * (n, c, h, w), contiguous; all reductions run in a fixed order (no float atomics), so every result is bit-reproducible
 * and an image's value does not depend on the rest of the batch.
 *
 * SSIM / MS-SSIM (metrics.py:37-63 gaussian_filter, 66-103 _ssim, 106-161 ssim, 164-236 ms_ssim): one hfc_ssim_level
 * launch per level, then one hfc_ssim_finalize.  (h0, w0) is the level-0 size; level l's inputs are (n, c, h_l, w_l),
 * h_{l+1} = (h_l + 1) / 2.  taps: (c, win) window taps per channel (odd win <= 31).  A dimension smaller than win is
 * not smoothed (the reference's gaussian_filter skips it).  c1 = (K1 * data_range)^2, c2 = (K2 * data_range)^2.
 * x_pooled / y_pooled: (n, c, h_{l+1}, w_{l+1}), the F.avg_pool2d(kernel 2, padding h_l % 2, w_l % 2) of x / y, the next
 * level's inputs; both NULL at the last level.  ws: device scratch of at least hfc_ssim_ws_bytes(n, c, h0, w0, win,
 * levels) bytes (8-byte aligned), shared by all levels of one call; it need not be initialised.
 * hfc_ssim_finalize: per plane, the mean over each level's valid outputs, relu(cs) below the last level, the last level's
 * ssim (relu'd when relu_last), prod_l value_l ** weights_host[l] (levels <= 8); out = the mean over all (n, c)
 * (size_average, out[0]) or per image (out[0..n)).  ms_ssim: relu_last = 1; ssim: levels = 1, weight 1,
 * relu_last = nonnegative_ssim.
 * --------------------------------------------------------------------------------------------------------- */
int64_t hfc_ssim_ws_bytes(int32_t n, int32_t c, int32_t h, int32_t w, int32_t win, int32_t levels);
int hfc_ssim_level(const float* x, const float* y, int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t level,
                   const float* taps, int32_t win, float c1, float c2, float* x_pooled, float* y_pooled, void* ws,
                   int64_t ws_bytes, void* stream);
int hfc_ssim_finalize(int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t win, int32_t levels, const float* weights_host,
                      int32_t relu_last, int32_t size_average, void* ws, int64_t ws_bytes, float* out, void* stream);
/* PSNR (metrics.py:7-18): out[i] = 20 log10(max_val) - 10 log10(mean over image i of (a - b)^2), fp64 throughout;
 * per_image = c * h * w.  ws: device scratch of at least hfc_psnr_ws_bytes(n, per_image) bytes.  Two launches. */
int64_t hfc_psnr_ws_bytes(int32_t n, int64_t per_image);
int hfc_psnr(const float* a, const float* b, int32_t n, int64_t per_image, double max_val, void* ws, int64_t ws_bytes,
             double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HFC_H_ */
