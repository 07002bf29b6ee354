/* cae_b200.h -- C ABI of the B200-native compress/decompress hot path.
 *
 * This is the drop-in boundary underneath the reference's Python surface.
 * The reference (TheJacksonLaboratory/cnn_autoencoder) has no FFI of its own:
 * its hot path is `torch.nn` modules plus CompressAI's C++ extension.  Each
 * entry point below names the reference call it replaces (paths relative to
 * the reference root, R = src/models/tasks/_autoencoders.py).  The host-side
 * mirror in cnn_autoencoder_b200/ (same class and function names as the
 * reference's `models` package) binds these with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions: plain pointers and sizes only (no torch types); the caller owns
 * every buffer; device pointers unless a parameter is marked HOST; every
 * device entry point takes the CUDA stream (a cudaStream_t passed as void*)
 * it enqueues on and returns without synchronising; return value 0 = ok,
 * otherwise an error code whose text cae_last_error() returns (thread-local).
 * There is no CPU fallback: a build without sm_100a code or a missing device
 * is an error, never a silent host path.
 */
#ifndef CAE_B200_H
#define CAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAE_ABI_VERSION 4

/* ---- tensor formats ------------------------------------------------------ */
enum {
  CAE_FMT_NONE = 0,
  CAE_FMT_U8_HWC = 1,     /* N x H x W x C uint8. As input: value/255.0f (R:545, compress.py:55);
                             as output: (uint8)clip(v*255,0,255), truncation (R:577-578).      */
  CAE_FMT_F32_NCHW = 2,   /* torch-contiguous fp32                                             */
  CAE_FMT_F16_PLANAR = 3, /* internal: [N][C/8][H+2][W+8][8] half, 1-pixel halo.  Padded pixel
                             (Y,X) = (y+1,x+1) is row Y, column X+3 (CAE_COL_PAD): pixel x=0
                             sits at column 4, so 8-channel units of a pixel run start on a
                             32-byte DRAM sector and every row is a whole number of sectors. */
  CAE_FMT_F16_SPLIT = 4   /* internal: [N][4][C/8][(H+2)/2][(W+8)/2][8] half; padded pixel
                             (Y,X) lives in parity plane (Y&1)*2+((X+3)&1) at (Y>>1,(X+3)>>1).
                             Feeds the stride-2 convolutions. H and W must be even.            */
};

#define CAE_COL_PAD 3     /* unused 16-byte units before the left halo column of a row */

enum { CAE_HALO_KEEP = 0,    /* leave the halo as allocated (zeros): zero padding (ConvTranspose2d) */
       CAE_HALO_REFLECT = 1  /* also write mirrored copies: padding_mode='reflect' (R:70,85)        */ };

enum { CAE_ACT_NONE = 0, CAE_ACT_LEAKY_RELU = 1 /* slope 0.01, R:26 */, CAE_ACT_RELU = 2 /* R:28 */ };

enum {
  CAE_CONV_S1 = 0,   /* nn.Conv2d k3 s1 p1            R:63-70, 114-121, 130-137              */
  CAE_CONV_S2 = 1,   /* nn.Conv2d k3 s2 p1            R:78-85, 148-155                        */
  CAE_CONVT_S1 = 2,  /* nn.ConvTranspose2d k3 s1 p1   R:189-196, 241-248, 258-265             */
  CAE_CONVT_S2 = 3   /* nn.ConvTranspose2d k3 s2 p1 output_padding 1   R:204-211, 278-285     */
};

enum { CAE_PAD_ZERO = 0, CAE_PAD_REFLECT = 1 };

typedef struct {
  void *ptr;
  int32_t fmt;      /* CAE_FMT_*                                                         */
  int32_t planes;   /* PLANAR/SPLIT: number of 8-channel planes (channels padded with 0) */
  int32_t halo;     /* outputs in PLANAR/SPLIT: CAE_HALO_*                                */
  int32_t reserved;
} cae_tensor;

/* One 3x3 (transposed) convolution with its fused epilogue:
 *   out = post_act( pre_act(conv(in) + bias) + skip )
 * which covers every unit of R:53-304 (bias R:41-42; activations R:19-34;
 * residual add R:172, R:302; image casts R:545, R:577-578).                    */
typedef struct {
  int32_t kind;            /* CAE_CONV_* */
  int32_t n, h_in, w_in;   /* batch and INPUT spatial size                               */
  int32_t c_in, c_out;     /* real channel counts                                        */
  cae_tensor in, out, skip;/* skip.fmt == CAE_FMT_NONE when absent; skip has out's size  */
  const void *weights;     /* igemm: packed (cae_pack_weights); direct: fp32 torch layout */
  const float *bias;       /* c_out floats or NULL                                       */
  int32_t pre_act, post_act;
  int32_t pad_mode;        /* direct kernel only (CAE_PAD_*); igemm reads the halo       */
  int32_t ck;              /* igemm: channels per K chunk (16/32/48/64/128 dividing c_in
                              padded to 16), 0 = auto; a ck whose activation stage and two
                              weight stages exceed shared memory is refused (e.g. 128 on a
                              stride-1 layer of 128 -> 192 channels, 64 on a stride-2 one)  */
  int32_t mt;              /* igemm: 16x8 M-tiles per CTA tile (1/2), 0 = auto           */
  int32_t grid;            /* igemm: CTAs, 0 = one per SM                                */
  void *aux_out;           /* optional second output (fp32 NCHW) or NULL                 */
  const struct cae_quant_fuse *quant; /* igemm + fp32 NCHW output (the latent layer) only:
                                         quantizer fused into the epilogue, or NULL      */
  int32_t groups;          /* direct kernel only: nn.Conv2d / nn.ConvTranspose2d `groups`
                              (the reference's groups=True builds every layer with
                              groups=channels_in, R:68, 83, 119, 135, 153); 0 or 1 = dense;
                              weights stay in torch layout (c_out, c_in/groups, 3, 3) resp.
                              (c_in, c_out/groups, 3, 3)                                 */
  int32_t reserved;
  const struct cae_proj_fuse *proj;   /* igemm, CAE_CONVT_S2 with 128 output channels only: the
                                         image layer that follows is folded in (below), or NULL */
} cae_conv_desc;

/* ---- library ------------------------------------------------------------- */
int cae_abi_version(void);
const char *cae_last_error(void);
/* sm count / compute capability of the current device; fails unless cc == 10.x */
int cae_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* number of kernels this library has launched in this process (bench "gpu_launches") */
uint64_t cae_launch_count(void);

/* ---- weights ------------------------------------------------------------- */
/* Bytes of the packed fp16 image of one layer's weights for the implicit-GEMM
 * kernel, and the packing itself (device -> device).  `w` is the fp32 tensor in
 * torch layout: Conv2d (c_out, c_in, 3, 3), ConvTranspose2d (c_in, c_out, 3, 3)
 * (SURVEY.md Appendix C).  `scale` (c_out floats or NULL) multiplies each output
 * channel (eval-mode BatchNorm folding, R:72-73).  ck as in cae_conv_desc.    */
size_t cae_packed_weight_bytes(int kind, int c_in, int c_out, int ck);
int cae_pack_weights(int kind, int c_in, int c_out, int ck, const float *w,
                     const float *scale, void *packed, void *stream);

/* ---- convolutions -------------------------------------------------------- */
/* tcgen05 / TMEM / TMA implicit-GEMM path (in: PLANAR for S1/CONVT, SPLIT for
 * CONV_S2, c_in padded to 16).  Replaces nn.Conv2d / nn.ConvTranspose2d forward
 * inside Analyzer.forward R:359-361 and Synthesizer.forward R:442-455.        */
int cae_conv_igemm(const cae_conv_desc *d, void *stream);
/* CUDA-core direct path for the thin image-side layers (c_in < 16: the 3->3
 * stem, R:63-70 with channels_org) and tiny nets; any format combination.
 * PLANAR / SPLIT outputs: the dense stride-1 form with c_in, c_out <= 4 (the tiled
 * stem) writes plane 0 only (its padded channels as +0) and leaves further planes
 * as allocated, so they must hold zeros (alloc_act clears them); every other form
 * writes all `planes`, padded channels as +0.                                    */
int cae_conv_direct(const cae_conv_desc *d, void *stream);

/* Fused head of an analysis track: the first DownsamplingUnit of the reference
 * (R:53-77: Conv2d(c_in, c_in, k3 s1) -> act -> Conv2d(c_in, c_out, k3 s2) [-> act],
 * called from Analyzer.forward R:359-361) in one launch,
 *   out = act_down( conv_s2( act_stem( conv_s1(in) + b_stem ) ) + b_down ).
 * The stem result stays in shared memory and feeds the tensor cores as an im2col
 * operand with K = 9 * c_in.  Weights are fp32 in torch Conv2d layout
 * (c_out, c_in, 3, 3) with any BatchNorm already folded; both convolutions use
 * `pad_mode`.  c_in 1..4, c_out <= 128.                                         */
typedef struct cae_head_desc {
  int32_t n, h_in, w_in;   /* input images                                        */
  int32_t c_in, c_out;
  cae_tensor in;           /* CAE_FMT_U8_HWC (x/255 applied) or CAE_FMT_F32_NCHW     */
  cae_tensor out;          /* CAE_FMT_F16_PLANAR, ceil(h/2) x ceil(w/2), halo KEEP/REFLECT */
  const float *w_stem;     /* [c_in][c_in][3][3]                                    */
  const float *b_stem;     /* [c_in] or NULL                                        */
  const float *w_down;     /* [c_out][c_in][3][3]                                   */
  const float *b_down;     /* [c_out] or NULL                                       */
  int32_t act_stem, act_down; /* CAE_ACT_*                                         */
  int32_t pad_mode;        /* CAE_PAD_*                                             */
  /* ResidualDownsamplingUnit (R:104-174) with a plain activation: the stem is
   *   fx = act_mid( conv_s1_b( act_stem( conv_s1_a(in) + b_stem ) ) + b_stem2 + in )
   * before the stride-2 convolution; residual = 0 selects the plain unit above.     */
  int32_t residual;
  const float *w_stem2;    /* [c_in][c_in][3][3] second stride-1 convolution, or NULL */
  const float *b_stem2;    /* [c_in] or NULL                                        */
  int32_t act_mid;         /* activation after the residual add                     */
  int32_t reserved;
} cae_head_desc;
int cae_conv_head(const cae_head_desc *d, void *stream);

/* Projection fusion of the last two synthesis layers (Synthesizer.forward R:442-455: the last
 * UpsamplingUnit's ConvTranspose2d(128, 128, k3 s2) -> act, then the image layer
 * ConvTranspose2d(128, c, k3 s2), c <= 3).  The image layer is linear in the 128-channel tensor U
 * between them, so the wide layer's epilogue multiplies each pixel of U with the image layer's
 * nine 128 x c tap matrices on the tensor cores and writes those 9 * c products (a 32 x fp16
 * record per pixel of U, `proj`: n x 2h x 2w x 32) instead of U itself (128 x fp16 per pixel);
 * cae_image_from_proj then adds the up to four records that meet in each output pixel, applies
 * bias / activations and writes the uint8 HWC image (truncating cast, R:577-578) and / or the
 * fp32 NCHW tensor.  U never reaches HBM.  h, w of cae_image_from_proj / cae_proj_bytes are the
 * size of U (twice the wide layer's input).  `scale` as in cae_pack_weights.                  */
typedef struct cae_proj_fuse {
  const void *weights;   /* cae_pack_proj_weights: cae_proj_weight_bytes() bytes */
  void *proj;            /* cae_proj_bytes(n, 2 * h_in, 2 * w_in) bytes          */
} cae_proj_fuse;
size_t cae_proj_weight_bytes(void);
size_t cae_proj_bytes(int n, int h, int w);
int cae_pack_proj_weights(int c_in, int c_out, const float *w /* (c_in, c_out, 3, 3) */,
                          const float *scale, void *packed, void *stream);
int cae_image_from_proj(const void *proj, int n, int h, int w, int c_out, const float *bias,
                        int pre_act, int post_act, void *out_u8, float *aux_nchw, void *stream);

/* ---- GDN / IGDN ---------------------------------------------------------- */
/* compressai.layers.GDN forward as used by _define_act_layer (R:29-30; SURVEY.md A.4):
 * out = x * rsqrt(beta + gamma . x^2)  (inverse: x * sqrt(...)), then "+ skip" when given
 * (the residual add of R:172 / R:302).  in/out/skip: PLANAR or SPLIT fp16, same H x W x C.
 * beta (c) and gamma (c x c, row i = output channel) are the re-parametrised fp32 values.  */
int cae_gdn(cae_tensor in, cae_tensor out, cae_tensor skip, int n, int h, int w, int c,
            const float *beta, const float *gamma, int inverse, void *stream);

/* ---- layout -------------------------------------------------------------- */
/* fp32 NCHW <-> internal planar fp16 (API boundary of Analyzer/Synthesizer). */
int cae_nchw_to_planar(const float *src, int n, int c, int h, int w, cae_tensor dst, void *stream);
int cae_planar_to_nchw(cae_tensor src, int n, int c, int h, int w, float *dst, void *stream);

/* ---- factorized-prior entropy model --------------------------------------- */
/* EntropyBottleneck.forward in eval mode + symbols + per-channel histogram
 * (CompressAI, reached from _taskutils.py:97 and R:549; SURVEY.md A.1):
 *   sym = rint(y - median_c); y_q = sym + median_c;
 *   p   = max(lut[c][sym - lut_min], 1e-9)   (exact per-(channel,symbol) table)
 *   hist[c][clamp(sym - hist_min, 0, hist_bins-1)] += 1
 *   rate_bits += sum(-log2 p)
 * y: fp32 N x C x hw.  Any output pointer may be NULL.  hist (C x hist_bins) and
 * rate_bits are ACCUMULATED into (zero them first).  Symbols outside the table
 * are evaluated with the density MLP; *status is set non-zero if that was needed
 * but no MLP was given.                                                        */
typedef struct cae_eb_tables {
  const float *medians;     /* C */
  const float *lut;         /* C x lut_len likelihoods (already lower-bounded) */
  int32_t lut_min, lut_len;
  /* density MLP for symbols outside the table (NULL = not provided: such symbols are an
   * error reported through `status`).  Per channel `mlp_stride` floats: for layer i of
   * n_layers: softplus(_matrix_i) [dims[i+1] x dims[i]], _bias_i [dims[i+1]], and, for
   * i < n_layers-1, tanh(_factor_i) [dims[i+1]].  dims = (1, filters..., 1).            */
  const float *mlp;
  int32_t n_layers, mlp_stride;
  int32_t dims[10];
  int32_t hist_min, hist_bins;
  /* > 0: the table reaches, on both sides, the symbols whose likelihood is the lower bound
   * (1e-9, CompressAI likelihood_bound), so every symbol outside the table has exactly this
   * likelihood and the MLP is never evaluated.  0: unknown, fall back to the MLP.            */
  float tail_lik;
  /* CompressAI's likelihood_lower_bound.bound (1e-9 unless the checkpoint says otherwise):
   * the floor applied to likelihoods evaluated on the device.                                */
  float lik_bound;
} cae_eb_tables;

int cae_eb_quantize(const float *y, int n, int c, int hw, const cae_eb_tables *t,
                    float *y_q, float *p_y, int32_t *symbols, int32_t *hist,
                    double *rate_bits, int32_t *status, void *stream);

/* EntropyBottleneck.decompress's de-quantisation ("symbols + medians", SURVEY.md A.1; reached from
 * R:568-572) written straight into the synthesis track's input layout: symbols int32
 * N x C x h x w -> dst planar fp16 (zero halo untouched), y_q = (float)sym + median_c.          */
int cae_eb_dequantize_planar(const int32_t *symbols, const float *medians, int n, int c, int h,
                             int w, cae_tensor dst, void *stream);

/* EntropyBottleneck.forward in TRAINING mode (additive-noise proxy + likelihood with gradients;
 * CompressAI, reached from _taskutils.py:97 inside the train step train_cae_ms.py:209-219;
 * SURVEY.md A.1), one fused kernel per direction instead of ~60 ATen launches:
 *   y_hat = y + noise;  l,u = logits_c(y_hat -+ 1/2);  s = -sign(l+u);
 *   lik = max(|sigmoid(s u) - sigmoid(s l)|, bound).
 * `blob` holds the EFFECTIVE per-channel parameters, C x cae_eb_train_blob_size() floats: for each
 * of the 5 layers of filters (3,3,3,3): softplus(_matrix_i) [dout x din], _bias_i [dout],
 * tanh(_factor_i) [dout] (none for the last layer) -- the caller keeps the softplus / tanh
 * Jacobians (tiny tensors).  Backward: given d/d y_hat and d/d lik (either may be NULL) writes
 * g_y = d/d y and ACCUMULATES d/d blob (zero it first); LowerBound passes the gradient where
 * the raw likelihood >= bound or the incoming gradient is negative.  noise may be NULL (0).   */
int cae_eb_train_blob_size(void);
int cae_eb_train_fwd(const float *y, const float *noise, const float *blob, int n, int c, int hw,
                     float bound, float *y_hat, float *lik, void *stream);
int cae_eb_train_bwd(const float *y_hat, const float *blob, int n, int c, int hw, float bound,
                     const float *g_yhat, const float *g_lik, float *g_y, float *g_blob,
                     void *stream);

/* ---- training: backward of the 3x3 (transposed) convolutions ---------------------------------
 * `loss.backward()` through nn.Conv2d / nn.ConvTranspose2d + activation of the units
 * (src/train_cae_ms.py:209-219 -> R:53-304).  Per layer, with z = conv(x) + b, out = act(z):
 *
 *  cae_act_grad   dz = fold(g) * act'(out) * scale, db += sum over pixels (unscaled).  g is the
 *                 gradient w.r.t. `out` as the next layer's data-gradient kernel left it; `fold`
 *                 adds the mirrored ring of a reflect-padded Conv2d consumer (g then covers the
 *                 PADDED input of that consumer: logical size g_h x g_w, pixel (0,0) of this
 *                 layer at (fold_shift + 1, fold_shift + 1)).  g / out / dz may each be fp32
 *                 NCHW, planar or split fp16; (oy, ox) place this layer's pixel (0,0) inside a
 *                 larger zero-ringed buffer (dz embedded for the data gradient of a reflect-padded
 *                 Conv2d: cae_conv_igemm of the TRANSPOSED kind on the embedded dz yields the
 *                 gradient of the padded input).  `scale` is a device scalar (loss scaling into
 *                 fp16 range) or NULL.
 *  data gradient  = cae_conv_igemm with the transposed kind on dz and the SAME weight tensor
 *                 (torch stores Conv2d weights as (out, in, 3, 3) and ConvTranspose2d weights
 *                 as (in, out, 3, 3), so cae_pack_weights(transposed kind, W) is the adjoint).
 *  cae_conv_wgrad dW += scale * sum_pixels dz (x) window(x) on the tensor cores (fp32, torch
 *                 layout, accumulated; up to 256 channels per side).  x: the layer's forward
 *                 input in the layout the forward kernel read (planar; split for CAE_CONV_S2);
 *                 dz: planar (split for CAE_CONVT_S2), zero halo; dz_embed = 1 when dz is
 *                 embedded as above.                                                          */
typedef struct cae_act_grad_desc {
  int32_t n, h, w, c;            /* the layer's OUTPUT: batch, size, channels                        */
  cae_tensor g;                  /* incoming gradient (fp32 NCHW, planar or split fp16)              */
  int32_t g_h, g_w, g_oy, g_ox;  /* logical size of g's buffer, position of pixel (0,0) in it        */
  int32_t fold, fold_shift;      /* fold = 1: g covers the reflect-padded input of the consumer      */
  cae_tensor out;                /* the layer's saved output (for the activation derivative), or none */
  int32_t out_h, out_w;
  int32_t act;                   /* activation between convolution and (optional) residual add       */
  int32_t post_act;              /* activation after the residual add (CAE_ACT_NONE / LEAKY_RELU)    */
  cae_tensor dz;                 /* result: gradient of the convolution's output                     */
  int32_t dz_h, dz_w, dz_oy, dz_ox;
  /* residual add (R:172, R:302: out = post_act(act(z) + skip)): `skip` = the tensor that was
   * added (h x w, the layout it was saved in); `gsum` (optional) receives g * post_act'(out), the
   * gradient that continues to the source of the skip; `g2` (optional, any layer) = such a
   * gradient arriving at THIS layer's output from a residual connection further up.            */
  cae_tensor skip, gsum, g2;
  const float *scale;            /* device scalar multiplied into dz / gsum, or NULL                 */
  float *db;                     /* c floats, accumulated (sums taken before `scale`), or NULL       */
} cae_act_grad_desc;
int cae_act_grad(const cae_act_grad_desc *d, void *stream);
size_t cae_conv_wgrad_workspace_bytes(void);   /* scratch for the per-CTA partial sums */
int cae_conv_wgrad(int kind, int n, int h_in, int w_in, int c_in, int c_out, cae_tensor x,
                   cae_tensor dz, int dz_embed, float *dw, const float *scale, void *workspace,
                   size_t workspace_bytes, void *stream);

/* The same quantizer fused into the epilogue of the last analysis convolution
 * (cae_conv_desc.quant; the layer whose output is the fp32 NCHW latent y, Analyzer.forward
 * R:359-361 followed by fact_ent R:549 / _taskutils.py:97): while y is still in registers the
 * epilogue also produces sym / y_q / the histogram / the rate exactly as cae_eb_quantize does
 * from y, and can write y_q in the planar fp16 layout the synthesis track reads, so the
 * latent makes one trip to HBM instead of three.  Every output may be NULL / CAE_FMT_NONE;
 * hist and rate_bits are accumulated into.                                       */
typedef struct cae_quant_fuse {
  cae_eb_tables tables;
  float *y_q;                /* fp32 NCHW                                          */
  int32_t *symbols;          /* int32 NCHW                                         */
  cae_tensor y_q_planar;     /* CAE_FMT_F16_PLANAR with planes = ceil(C/16)*2, zero halo */
  int32_t *hist;             /* C x tables.hist_bins                                */
  double *rate_bits;
  int32_t *status;
} cae_quant_fuse;

/* ---- entropy coder (HOST, thread-safe, no globals) ------------------------ */
/* compressai._CXX.pmf_to_quantized_cdf (SURVEY.md A.2), reached from
 * EntropyBottleneck.update R:502, R:615.  cdf has n+1 entries.                */
int cae_pmf_to_quantized_cdf(const float *pmf /*HOST*/, int n, int precision,
                             uint32_t *cdf /*HOST*/);
/* compressai.ans.RansEncoder.encode_with_indexes / RansDecoder.decode_with_indexes
 * (SURVEY.md A.3) for the EntropyBottleneck index pattern: `symbols` is C-major
 * raster (C x hw), symbol i uses table i / hw.  Reached from R:549-551, 568-572,
 * 645-647, 662-665.  cdfs: C x cdf_stride int32.  Returns 0 and *nbytes.      */
int cae_rans_encode(const int32_t *symbols /*HOST*/, int c, int hw, const int32_t *cdfs,
                    int cdf_stride, const int32_t *cdf_sizes, const int32_t *offsets,
                    uint8_t *out /*HOST*/, size_t out_cap, size_t *nbytes);
int cae_rans_decode(const uint8_t *enc /*HOST*/, size_t nbytes, int c, int hw,
                    const int32_t *cdfs, int cdf_stride, const int32_t *cdf_sizes,
                    const int32_t *offsets, int32_t *symbols /*HOST*/);

/* ---- entropy coder (DEVICE, batched: one thread per tile stream, symbols staged per warp) ------------ */
/* Same stream format as cae_rans_encode / cae_rans_decode, for n independent streams at once
 * (the tiles of a slide; SURVEY.md 8f-1).  symbols: n x C x hw int32.  Encoding writes stream k
 * into the TAIL of words[k*cap_words .. (k+1)*cap_words) and its length into nwords[k]
 * (cap_words >= C*hw + 64 is always enough short of pathological escape counts; overflow sets
 * bit 0 of *status).  cae_rans_compact packs the tails back to back at out_offsets[k] (an
 * exclusive prefix sum of nwords, in words).  Decoding reads stream k from
 * words[word_offsets[k] .. word_offsets[k+1]) (bit 1 of *status: a stream was truncated).
 * All pointers are device pointers; tables as in the host entry points.                   */
/* Optional per-(channel, symbol) encode table (16 bytes per entry, C x cdf_stride entries on the
 * device) that replaces the 64-bit division of the state update by an exact reciprocal
 * multiply; built once per set of CDFs.  enc_table == NULL encodes with the plain division.   */
size_t cae_rans_enc_table_bytes(int c, int cdf_stride);
int cae_rans_build_enc_table(const int32_t *cdfs, int c, int cdf_stride, const int32_t *cdf_sizes,
                             void *table, void *stream);
int cae_rans_encode_batch(const int32_t *symbols, int n, int c, int hw, const int32_t *cdfs,
                          int cdf_stride, const int32_t *cdf_sizes, const int32_t *offsets,
                          const void *enc_table, uint32_t *words, int cap_words, int32_t *nwords,
                          int32_t *status, void *stream);
/* out_offsets[0..n] = exclusive prefix sum of nwords (out_offsets[n] = total words), on the
 * device, so that packing needs no host round trip.                                        */
int cae_rans_scan(const int32_t *nwords, int n, int64_t *out_offsets, void *stream);
int cae_rans_compact(const uint32_t *words, int n, int cap_words, const int32_t *nwords,
                     const int64_t *out_offsets, uint32_t *out, void *stream);
int cae_rans_decode_batch(const uint32_t *words, const int64_t *word_offsets, int n, int c, int hw,
                          const int32_t *cdfs, int cdf_stride, const int32_t *cdf_sizes,
                          const int32_t *offsets, int32_t *symbols, int32_t *status, void *stream);

/* ---- tile-loop front end (HOST, native threads) ------------------------------- */
/* What the reference leaves to dask's threaded scheduler and zarr's chunk store
 * (compress.py:101-128, decompress.py:72-96), on whole batches of tiles so that a Python loop
 * does not bound the GPU.  All pointers are host pointers; `threads` native threads per call.
 *  cae_tiles_gather_u8: dst[k] = ps x ps x c tile (tile_yx[2k], tile_yx[2k+1]) of the row-major
 *    H x W x c uint8 image, edge tiles zero filled (zarr's chunk padding).
 *  cae_files_write: file k = headers[k*hdr_len ..][hdr_len] + payload[payload_off[k] ..
 *    payload_off[k+1]); paths = n NUL-terminated strings back to back; written as
 *    <path>.partial then renamed.
 *  cae_files_stat / cae_files_read: sizes, then header / payload split back the same way.
 *  cae_files_remove: unlink n files (missing ones are skipped) -- the chunks of an array that
 *    is created again with overwrite=True (compress.py:123-128, decompress.py:92-96).       */
int cae_tiles_gather_u8(const uint8_t *src, int64_t H, int64_t W, int c, int ps,
                        const int32_t *tile_yx, int n, uint8_t *dst, int threads);
int cae_files_write(const char *paths, int n, const uint8_t *headers, int hdr_len,
                    const uint8_t *payload, const int64_t *payload_off, int threads);
int cae_files_stat(const char *paths, int n, int64_t *sizes, int threads);
int cae_files_remove(const char *paths, int n, int threads);
int cae_files_read(const char *paths, int n, uint8_t *headers, int hdr_len, uint8_t *payload,
                   const int64_t *payload_off, int threads);

/* ---- tile movement between the host slide and the device (strided DMA) ---------------------- */
/* The chunk loop of compress.py:101-128 / decompress.py:72-96 without a host-side gather: tile k
 * = (tile_yx[2k], tile_yx[2k+1]) of the row-major H x W x c uint8 slide in HOST memory (page-locked
 * for the copies to be asynchronous) <-> slot k of a tile-major DEVICE buffer n x ps x ps x c,
 * enqueued on `stream`.  Upload zero-fills the part of an edge tile beyond the image (zarr's
 * chunk padding), download crops it.  tile_yx is a HOST array.                                */
int cae_tiles_upload_u8(const uint8_t *src /*HOST*/, int64_t H, int64_t W, int c, int ps,
                        const int32_t *tile_yx /*HOST*/, int n, uint8_t *dst, void *stream);
int cae_tiles_download_u8(const uint8_t *src, int n, int ps, int c, const int32_t *tile_yx /*HOST*/,
                          uint8_t *dst /*HOST*/, int64_t H, int64_t W, void *stream);

/* The same with tiles that sit side by side in one tile row of the slide moved as ONE copy of the
 * band segment (rows of r * ps * c bytes instead of ps * c: the DMA engines reach the link's
 * contiguous rate) and re-tiled on the device; `scratch`: device buffer of n * ps * ps * c bytes.
 * Isolated and edge tiles take the per-tile copies above.                                      */
int cae_tiles_upload_u8_banded(const uint8_t *src /*HOST*/, int64_t H, int64_t W, int c, int ps,
                               const int32_t *tile_yx /*HOST*/, int n, uint8_t *dst,
                               uint8_t *scratch, void *stream);
int cae_tiles_download_u8_banded(const uint8_t *src, int n, int ps, int c,
                                 const int32_t *tile_yx /*HOST*/, uint8_t *dst /*HOST*/, int64_t H,
                                 int64_t W, uint8_t *scratch, void *stream);

/* Region reads: windows cut out of one batch of decoded tiles, on the device.  `tiles`: tile-major
 * n_tiles x ps x ps x c; `out`: n_boxes x box_h x box_w x c.  Piece i = pieces[8i .. 8i+7] =
 * {k, b, sy, sx, dy, dx, h, w}: rows [sy, sy+h) x columns [sx, sx+w) of tile k go to (dy, dx) of
 * box b; k = -1 writes zeros instead (the fill value of a chunk whose file is missing).  Every
 * piece is checked on the host before the table is copied to `pieces_dev` (DEVICE, m x 8 int32,
 * 16-byte aligned) on `stream`; one launch copies them all.                                    */
int cae_tiles_crop_u8(const uint8_t *tiles, int n_tiles, int ps, int c,
                      const int32_t *pieces /*HOST, m x 8*/, int m, int32_t *pieces_dev /*m x 8*/,
                      uint8_t *out, int n_boxes, int box_h, int box_w, void *stream);

/* Region writes: the inverse.  The same piece table, read the other way: rows [dy, dy+h) x columns
 * [dx, dx+w) of box b of `boxes` (n_boxes x box_h x box_w x c) go to (sy, sx) of tile k of `tiles`;
 * b = -1 writes zeros instead (the padding of an edge chunk; dy, dx are then ignored).  The pieces
 * of one call must not overlap in `tiles`.  Checked on the host like cae_tiles_crop_u8; bytes of
 * `tiles` outside the pieces are left as they are.                                             */
int cae_tiles_paste_u8(uint8_t *tiles, int n_tiles, int ps, int c,
                       const int32_t *pieces /*HOST, m x 8*/, int m, int32_t *pieces_dev /*m x 8*/,
                       const uint8_t *boxes, int n_boxes, int box_h, int box_w, void *stream);

/* Reduced-resolution region reads: windows of the level-f image cut out of one batch of decoded
 * tiles.  f is a power of two in [1, 512] that divides ps; level pixel (i, j) of tile k, channel
 * ch, is the mean, rounded half up ((s + n/2) / n over the n pixels), of level-0 rows
 * [i f, min((i+1) f, vh)) x columns [j f, min((j+1) f, vw)) of the tile.  Piece i =
 * pieces[12i .. 12i+11] = {k, b, sy, sx, dy, dx, h, w, vh, vw, 0, 0}: the crop's record in level
 * pixels (tile k's level grid is (ps/f)^2; `out` is n_boxes x box_h x box_w x c level pixels) and
 * the in-array extent 0 < vh, vw <= ps of tile k in level-0 pixels (ps, except for edge chunks;
 * the padding beyond it never enters a mean; (sy+h-1) f < vh and (sx+w-1) f < vw).  k = -1 writes
 * zeros.  Checked on the host like cae_tiles_crop_u8; `pieces_dev`: DEVICE, m x 12 int32,
 * 16-byte aligned.                                                                             */
int cae_tiles_crop_reduce_u8(const uint8_t *tiles, int n_tiles, int ps, int c, int f,
                             const int32_t *pieces /*HOST, m x 12*/, int m,
                             int32_t *pieces_dev /*m x 12*/, uint8_t *out, int n_boxes, int box_h,
                             int box_w, void *stream);

/* Resolution pyramid: levels 1..K (1 <= K <= 9, 2^K divides ps) of one batch of decoded tiles in
 * one launch, each tile read once.  recs[4t .. 4t+3] = {i, j, vh, vw}: tile t is chunk (i, j) of
 * a gy x gx level-0 chunk grid, with in-array extent 0 < vh, vw <= ps.  `out` holds one chunk row
 * of every level, level after level: level k is ceil(gx / 2^k) tile-major ps x ps x c tiles,
 * starting at tile sum_{l<k} ceil(gx / 2^l).  Tile t's level-k pixels (the means of
 * cae_tiles_crop_reduce_u8 at f = 2^k: rounded half up, over level-0 pixels inside vh x vw only)
 * go to tile j >> k of level k at rows (i mod 2^k) ps/2^k + [0, ceil(vh/2^k)) and columns
 * (j mod 2^k) ps/2^k + [0, ceil(vw/2^k)); no other byte of `out` is written.  The tiles of one
 * call must be distinct chunks of one level-1 chunk row (equal i >> 1).  Checked on the host like cae_tiles_crop_u8; `recs_dev`: DEVICE,
 * n_tiles x 4 int32, 16-byte aligned.                                                          */
int cae_tiles_pyramid_u8(const uint8_t *tiles, int n_tiles, int ps, int c, int levels,
                         const int32_t *recs /*HOST, n_tiles x 4*/, int32_t *recs_dev, int gy,
                         int gx, uint8_t *out, void *stream);

/* ---- evaluation sums on the device (SURVEY.md 8f-4) ------------------------------------------ */
/* sse[i] += sum over the per_image uint8 values of image i of (a - b)^2: the numerator of
 * compute_rmse / compute_psnr (src/test_cae.py:57-63, computed there on the host after a full
 * download) and of DistMSELoss in uint8 units (_ratedist.py:57-63).  a, b: n_images x per_image
 * uint8 on the device; sse: n_images uint64 on the device, accumulated into.                   */
int cae_sse_u8(const uint8_t *a, const uint8_t *b, int n_images, int64_t per_image,
               uint64_t *sse, void *stream);

/* skimage.metrics.structural_similarity(x, x_r, channel_axis=2) with its defaults, as
 * compute_ssim calls it (src/test_cae.py:52-54): 7x7 uniform window, K1 0.01, K2 0.03, sample
 * covariance, data range 255.  a, b: n_images x h x w x c uint8 on the device; sum[i] += the SSIM
 * map of image i summed over the (h - 6) x (w - 6) window positions skimage keeps (its crop by 3)
 * and over the channels; SSIM = sum / ((h - 6)(w - 6) c).                                       */
int cae_ssim_u8(const uint8_t *a, const uint8_t *b, int n_images, int h, int w, int c, double *sum,
                void *stream);
/* compute_deltaCIELAB (src/test_cae.py:21-44): skimage.color.rgb2lab of both 8-bit sRGB images
 * (D65, 2 degree observer) and deltaE_cie76; sum[i] += the per-pixel colour distances of image i
 * (n_images x pixels x 3 uint8); mean = sum / pixels.                                           */
int cae_delta_e_u8(const uint8_t *a, const uint8_t *b, int n_images, int64_t pixels, double *sum,
                   void *stream);

/* Building blocks of compute_ms_ssim (src/test_cae.py:46-50: pytorch_msssim.ms_ssim(x_r, x,
 * data_range=255) with its defaults -- 11-tap Gaussian window, sigma 1.5, five scales, weights
 * 0.0448 0.2856 0.3001 0.2363 0.1333), all on fp32 planes [planes][h][w] on the device:
 *  cae_u8_to_planes_f32        N x H x W x C uint8 -> N * C planes
 *  cae_ssim_gauss_planes_f32   per plane, sum over the (h - 10) x (w - 10) valid window positions
 *                              of the SSIM map and of the contrast-structure map (accumulated)
 *  cae_avgpool2_planes_f32     F.avg_pool2d(x, 2, padding = size % 2): the next scale,
 *                              ((h + 2 (h % 2) - 2) / 2 + 1) x (same for w)
 * metrics.ms_ssim combines the five scales (relu, weighted product, mean over planes).          */
int cae_u8_to_planes_f32(const uint8_t *src, int n, int h, int w, int c, float *dst, void *stream);
int cae_avgpool2_planes_f32(const float *src, int planes, int h, int w, float *dst, void *stream);
int cae_ssim_gauss_planes_f32(const float *a, const float *b, int planes, int h, int w,
                              float data_range, double *sum_ssim, double *sum_cs, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CAE_B200_H */
