/* udb.h -- C ABI of libudb.so: the sm_100a kernels behind unidepth_b200's UniDepthV2.infer().
 *
 * The reference (lpiccinelli-eth/UniDepth) has no FFI on its inference path: every op below
 * replaces a PyTorch library call made by the reference's Python (file:line cited per entry,
 * relative to the reference repo root).  The Python host (unidepth_b200/) binds these with ctypes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller (PyTorch's
 *     caching allocator) owns all memory, the library never allocates, frees, copies to the host
 *     or synchronises the device;
 *   - every launch goes to the `stream` argument (a cudaStream_t passed as void*), so calls are
 *     CUDA-graph capturable;
 *   - return value 0 = OK; non-zero = error, message via udb_last_error() (thread-local);
 *   - "f16" tensors are IEEE half, "f32" are float; activations that feed tensor-core GEMMs are
 *     f16, residual streams / LayerNorm statistics / softmax / epilogue math are f32.
 */
#ifndef UDB_H_
#define UDB_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UDB_VERSION 1

int udb_version(void);

/* Per-launch profile: between begin and end every kernel this library enqueues on `stream` is followed by a CUDA event;
 * end synchronises and returns, per launch in order, the kernel's name, the time since the previous event (its duration
 * when the stream stays busy) and the algorithmic flops / bytes its launcher declared.  Returns the number of launches
 * (which may exceed cap; only the first cap entries are written), -1 on error.  Not for use under stream capture. */
typedef struct udb_profile_entry_t {
  char name[48];
  float ms;
  double flops;
  double bytes;
} udb_profile_entry_t;
int udb_profile_begin(void* stream);
int udb_profile_end(udb_profile_entry_t* out, int32_t cap);
const char* udb_last_error(void);
/* Number of kernels launched by this library on the calling process since load (bench evidence). */
int64_t udb_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core GEMM  D = epilogue(A . W^T)  (tcgen05.mma kind::f16, fp32 accumulation in TMEM, TMA
 * operand loads, persistent warp-specialised kernel).
 * Replaces nn.Linear / nn.Conv2d(k=s=14) / nn.Conv2d(1x1, 3x3) / nn.ConvTranspose2d(k=s) calls:
 *   unidepth/models/backbones/metadinov2/{patch_embed.py:82, attention.py:55-61, mlp.py:36-40},
 *   unidepth/layers/{attention.py:119-138, mlp.py:29-34, upsample.py:171-180,218-222},
 *   unidepth/models/unidepthv2/decoder.py:43,264,279,288-303.
 * ------------------------------------------------------------------------------------------- */
enum { UDB_A_MATRIX = 0, UDB_A_CONV3X3 = 1 };
enum { UDB_ACT_NONE = 0, UDB_ACT_GELU = 1, UDB_ACT_LEAKY = 2 };
enum { UDB_STORE_ROWS = 0, UDB_STORE_CONVT = 1, UDB_STORE_CONVTILE = 2, UDB_STORE_HEAD = 3 };

typedef struct udb_gemm_t {
  /* operands: A f16 [M,K] row-major (lda elements) or NHWC f16 image for UDB_A_CONV3X3;
   * W f16 [N,K] row-major (ldw elements).  K-extent is zero-extended to a multiple of 64. */
  const void* a;
  const void* w;
  int32_t M, N, K;
  int32_t lda, ldw;
  int32_t a_mode;
  /* UDB_A_CONV3X3: input [B, H(+2), W(+2), C] f16 NHWC; K = 9*C ordered (dy,dx,c); the output
   * pixel (y,x) reads input (y+dy+off, x+dx+off), off = -1 for zero padding (out-of-range taps
   * read 0 through TMA out-of-bounds fill) or 0 when the input was padded by the caller
   * (reflect padding, in_H = H+2, in_W = W+2). */
  int32_t conv_B, conv_H, conv_W, conv_C, conv_inH, conv_inW, conv_off, conv_TH, conv_TW;
  /* the input may be a channel slice [conv_coff, conv_coff + conv_C) of a wider NHWC buffer with
   * conv_cstride channels per pixel (0 = conv_C) */
  int32_t conv_cstride, conv_coff;
  /* epilogue: v = acc + bias[n]; v = act(v); v *= gamma[n]; v += resid[...]; out = v;
   * out2 = f16(v) or f16(leaky(v)) (optional second f16 copy, e.g. the next conv's input) */
  const float* bias;
  const float* gamma;
  const void* resid;
  int32_t resid_f32; /* 1: f32, 0: f16 */
  void* out;
  int32_t out_f32;
  void* out2;
  int32_t out2_leaky; /* 1: out2 = f16(leaky(v)); 0: out2 = f16(v) */
  int32_t act;
  int32_t store_mode;
  int64_t ldc; /* elements between consecutive output rows / pixels */
  /* UDB_STORE_ROWS: out_row = (m / rows_per_group)*group_stride + m % rows_per_group + row_offset
   * (rows_per_group <= 0: identity).  resid row = resid_mod > 0 ? m % resid_mod + resid_row_offset
   * : out_row, with leading dimension ldr. */
  int32_t rows_per_group, group_stride, row_offset;
  int32_t resid_mod, resid_row_offset;
  int64_t ldr;
  /* UDB_STORE_CONVT: row m = (b, y, x) of a [B,h,w] grid; column n = (dy*k+dx)*Cout + co;
   * writes NHWC pixel (b, y*k+dy+pad, x*k+dx+pad, co) of a [B, h*k+2*pad, w*k+2*pad, Cout] map
   * (pad > 0: the interior of a buffer whose border udb_reflect_border_fill_nhwc_f16 fills). */
  int32_t ct_k, ct_cout, ct_h, ct_w, ct_pad;
  /* UDB_STORE_HEAD (N == 32): out_pixel = exp(clamp(sum_n head_w[n]*leaky(acc+bias)[n] + head_b,
   * -8, 8) + head_add) written as f32 to out[b*H*W + y*W + x]. */
  const float* head_w;
  float head_b, head_add;
  /* Split-f16 ("precise") operands, UDB_A_MATRIX only.  a_split_k = K1 > 0: every A row holds [hi(K1) | lo(K1)] with
   * x = hi + lo to ~22 bits (lo = f16(x - f32(hi))), lda >= 2*K1; W is packed [N, 3*K1] = [W_hi | W_hi | W_lo];
   * K must be 3*K1.  The k-blocks of the third segment re-read A's hi half, so the same MMAs accumulate
   * hi.W_hi + lo.W_hi + hi.W_lo in f32 -- the f16 product error (2^-11 per operand) drops to ~2^-21.
   * out_split > 0 (f16 `out`): also store lo = f16(v - f32(hi)) at column n + out_split, i.e. the output is itself a
   * split operand for the next GEMM. */
  int32_t a_split_k;
  int32_t out_split;
  /* Fused LayerNorm (the north_star's "fused LayerNorm + QKV projection"; reference metadinov2/block.py:84-109: the
   * LayerNorm that follows a residual update never runs as its own pass).
   * PRODUCER (ln_stats_out != NULL, ROWS store): besides its normal outputs the GEMM writes, for every output row and
   * every (column tile, column half) part, float2 {mean, centred sum of squares} of the values it stored:
   * ln_stats_out[(row * ln_parts + part)], ln_parts = (N / tile width) * 2, ln_part_cols = tile width / 2 (the call
   * fails if the caller's ln_parts / ln_part_cols do not match the tiling).  Use out2 for the f16 copy of the rows.
   * CONSUMER (ln_stats_in != NULL): A is that un-normalised f16 copy, W holds W * diag(ln_weight); the epilogue merges the
   * row's parts into mean / rstd (eps = ln_eps) and computes rstd * (acc - mean * ln_c1[n]) + bias[n], with
   * ln_c1[n] = sum_k W'[n,k] and bias = W ln_bias + linear bias -- algebraically LayerNorm followed by the Linear. */
  float* ln_stats_out;
  const float* ln_stats_in;
  const float* ln_c1;
  int32_t ln_parts, ln_part_cols;
  float ln_eps;
} udb_gemm_t;

int udb_gemm_f16(const udb_gemm_t* g, void* stream);

/* ---------------------------------------------------------------------------------------------
 * 3x3 convolution with few output channels over a PRE-PADDED NHWC f16 image [B, H+2, W+2, cstride]
 * (channel slice [coff, coff+C)), weights f16 [Cout, 9*C] ordered (dy,dx,c), Cout in {32, 64}.
 * The input halo of each 16x8-pixel tile is loaded once and shared by the nine taps (shifted UMMA
 * descriptors); weights stay resident in shared memory.  out: f16 NHWC [B,H,W,ldc] -- or, with
 * head_out != NULL (Cout == 32), the fused head exp(clamp(sum_n head_w[n]*act(conv)[n] + head_b,
 * -8, 8) + head_add) as an f32 plane [B,H,W].  Replaces the reflect-padded nn.Conv2d calls of
 * unidepth/models/unidepthv2/decoder.py:200-229 (to_depth_lr/hr, to_confidence_lr/hr).
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_conv_halo_t {
  const void* x;
  const void* w;
  const float* bias;
  int32_t B, H, W, C, cstride, coff, cout, act;
  void* out;
  int64_t ldc;
  const float* head_w;
  float head_b, head_add;
  float* head_out;
} udb_conv_halo_t;
int udb_conv3x3_halo_f16(const udb_conv_halo_t* c, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused softmax(Q K^T / sqrt(d)) V  (flash-style, tcgen05 QK^T and PV, S/O accumulators in TMEM).
 * Replaces F.scaled_dot_product_attention: metadinov2/attention.py:58, layers/attention.py:136.
 * q/k/v are f16 matrices with row stride ld* (elements); head h occupies columns
 * [col0 + h*head_dim, +head_dim).  Row of (batch b, position s) = b*seq + s.  out f16 [B*Sq, ldo].
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_attn_t {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int32_t B, heads, seq_q, seq_k, head_dim;
  int32_t ldq, ldk, ldv, ldo;
  int32_t q_col0, k_col0, v_col0, o_col0;
  float scale; /* 1/sqrt(head_dim) */
  /* Split-f16 ("precise") mode: when split != 0 the lo halves of q / k / v / out live lo_off_* elements to the right of
   * the hi halves (value = hi + lo) and the attention runs in an fp32 CUDA-core kernel (exact exp, f32 products):
   * a debugging / parity mode, ~50x slower than the tcgen05 kernel. */
  int32_t split;
  int32_t lo_off_q, lo_off_k, lo_off_v, lo_off_o;
} udb_attn_t;

int udb_attention_f16(const udb_attn_t* a, void* stream);

/* ---------------------------------------------------------------------------------------------
 * LayerNorm over the last dim (F.layer_norm): metadinov2/block.py:86,89 (eps 1e-6),
 * dinov2.py:336-345 (final norm, eps 1e-5), layers/attention.py:116-117, layers/mlp.py:30,
 * unidepthv2/decoder.py:190-199.  Input row r is read from in + in_row(r)*ld_in with
 * in_row(r) = (r / rows_per_group)*group_stride + r % rows_per_group + row_offset (identity if
 * rows_per_group <= 0) -- used to drop / pick the cls token of each image.
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_layernorm_t {
  const void* in;
  int32_t in_f32;
  void* out;
  int32_t out_f32;
  const float* weight;
  const float* bias;
  int32_t rows, dim;
  int64_t ld_in, ld_out;
  int32_t rows_per_group, group_stride, row_offset;
  float eps;
  int32_t dim_valid; /* 0 = dim.  f16->f16 rows of 64/128/256 only: statistics over the first dim_valid
                        columns (zero-padded channel rows, e.g. ViT-B's 96-channel map stored as 128) */
  int32_t out_split; /* > 0 (f32 -> f16 rows only): also store lo = f16(y - f32(hi)) at column + out_split */
} udb_layernorm_t;

int udb_layernorm(const udb_layernorm_t* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pre-processing + patch extraction (unidepthv2.py:288-297 + patch_embed.py:82's im2col):
 * uint8 (or f32 0..255) NCHW -> /255 -> (x-mean)/std -> zero pad -> bilinear (align_corners=False)
 * to (net_h, net_w) -> f16 patch matrix [B*gh*gw, ldp] with column c*196 + py*14 + px
 * (columns >= 588 zero).
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_preprocess_t {
  const void* rgb;
  int32_t rgb_is_u8; /* 1: uint8, 0: float32 */
  int32_t normalize;
  int32_t B, H, W;
  int32_t pad_l, pad_r, pad_t, pad_b;
  int32_t net_h, net_w;
  void* patches;
  int32_t ldp;
  int32_t split; /* 1: rows hold [hi | lo] halves of ldp/2 columns each (split-f16 precise mode) */
} udb_preprocess_t;

int udb_preprocess_patchify(const udb_preprocess_t* p, void* stream);

/* Bicubic (A=-0.75, align_corners=False, no antialias) resize of the [1,M,M,D] position grid to
 * [gh,gw,D] (dinov2.py:267-304, interpolate_offset == 0).  f32 -> f32. */
int udb_posembed_bicubic(const float* grid, int32_t m, int32_t dim, float* out, int32_t gh,
                         int32_t gw, void* stream);

/* x[b, 0, :] = cls_token + pos_embed[0]   (dinov2.py:314-315); x f32 [B, T, D]. */
int udb_set_cls_rows(float* x, const float* cls_token, const float* pos0, int32_t B, int32_t T,
                     int32_t D, void* stream);
/* Same, for the fused-LayerNorm encoder (udb_gemm_t.ln_*): also writes the f16 copy of the cls rows and their per-part
 * {mean, centred sum of squares} (parts * part_cols == D, the producer GEMMs' tiling). */
int udb_set_cls_rows_ln(float* x, void* x16, float* stats, const float* cls_token, const float* pos0, int32_t B, int32_t T,
                        int32_t D, int32_t parts, int32_t part_cols, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Small fp32 dense layer for the 4-token camera head (unidepthv2/decoder.py:101-111), kept in
 * fp32 on CUDA cores to protect the 1e-4 intrinsics bar:
 *   y[m, n] = resid[m,n] + gamma[n] * act(sum_k x[m,k] * w[n,k] + bias[n])      M <= 64
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_small_linear_t {
  const float* x;
  const float* w;
  const float* bias;
  const float* gamma;
  const float* resid;
  float* y;
  int32_t M, N, K;
  int32_t act;
  int32_t ldx, ldy, ldr; /* row strides (elements) of x, y, resid; 0 = dense (K, N, N) */
} udb_small_linear_t;
int udb_small_linear_f32(const udb_small_linear_t* p, void* stream);

/* Self-attention over the 4 camera tokens, fp32 (layers/attention.py:110-138 with pos_embed added
 * to q only).  q [B,4,C], kv [B,4,2C] (k then v), pos [4,C] -> out [B,4,C]. */
int udb_camera_attn4_f32(const float* q, const float* kv, const float* pos, float* out, int32_t B,
                         int32_t C, int32_t heads, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Camera tail + rays (unidepthv2/decoder.py:85-99, 361-403; utils/coordinate.py:4-20):
 *   x[B,4] -> (fx,fy,cx,cy) = (exp,exp,sigmoid,sigmoid) * (0.7*diag, 0.7*diag, W, H)
 *   K_net[B,3,3]; K_out[B,3,3] = post-processed (unidepthv2.py:92-108); intr4[B,4].
 * ------------------------------------------------------------------------------------------- */
int udb_camera_intrinsics(const float* x, int32_t B, int32_t net_h, int32_t net_w, float factor,
                          int32_t pad_l, int32_t pad_t, float* intr4, float* k_net, float* k_out,
                          void* stream);

/* Ray embedding (unidepthv2/decoder.py:234-253; utils/geometric.py:227-252;
 * utils/positional_embedding.py:218-256): unit rays from intr4 (or from rays_in [B,net_h*net_w,3]
 * when not NULL) -> antialiased bilinear down-sample by `net/grid` -> renormalise -> polar,
 * azimuth -> sin(angle * pi * scales[j]); out f32/f16 [B*gh*gw, 2*bands]. */
/* infer(camera=K) (unidepthv2.py:267-303; Camera.crop / resize utils/camera.py:78-81,115-120):
 * K [B,3,3] pinhole in input-image pixels -> (fx,fy,cx,cy) in network-input pixels. */
int udb_camera_adjust_k(const float* K, int32_t B, float factor, int32_t pad_l, int32_t pad_t,
                        float* intr4, void* stream);

typedef struct udb_ray_embed_t {
  const float* intr4;
  const float* rays_in;
  const float* scales; /* [bands] */
  int32_t B, net_h, net_w, gh, gw, bands;
  void* out;
  int32_t out_f32;
} udb_ray_embed_t;
int udb_ray_embed(const udb_ray_embed_t* p, void* stream);

/* x2 bilinear up-sample, align_corners=False (layers/upsample.py:215), NHWC f16 -> f16.
 * Optionally fused: out = up(x) is followed by nothing; see udb_gemm for the convT add. */
int udb_upsample2x_nhwc_f16(const void* in, void* out, int32_t B, int32_t H, int32_t W, int32_t C,
                            void* stream);

/* Bilinear align_corners=True resize NHWC f16 [B,H,W,C] -> [B,oh,ow,C] written into a buffer
 * reflect-padded by `pad` pixels on each side ([B,oh+2*pad,ow+2*pad,C]); pad = 0 gives the plain
 * resize (unidepthv2/decoder.py:299-301 + the reflect pad of the following conv :207-219). */
int udb_resize_ac_pad_nhwc_f16(const void* in, void* out, int32_t B, int32_t H, int32_t W,
                               int32_t C, int32_t oh, int32_t ow, int32_t pad, void* stream);

/* Reflect-pad by 1 pixel: NHWC f16 [B,H,W,C] -> [B,H+2,W+2,C] (nn.Conv2d padding_mode="reflect",
 * unidepthv2/decoder.py:200-213). */
int udb_reflect_pad1_nhwc_f16(const void* in, void* out, int32_t B, int32_t H, int32_t W, int32_t C,
                              void* stream);

/* Fill the 1-pixel border of a padded NHWC f16 buffer [B,H+2,W+2,C] by reflection of its interior
 * (the interior having been written by a GEMM with ct_pad = 1). */
int udb_reflect_border_fill_nhwc_f16(void* buf, int32_t B, int32_t H, int32_t W, int32_t C, void* stream);

/* =============================================================================================
 * UniDepthV1 operators (ConvNeXt encoder + V1 decoder; BASELINE config 4).  Reference call sites:
 * unidepth/models/backbones/convnext.py:130-298,459-471, unidepth/models/unidepthv1/decoder.py:38-300,
 * unidepth/models/unidepthv1/unidepthv1.py:30-94,288-373, unidepth/layers/{convnext,upsample,nystrom_attention}.py,
 * unidepth/utils/geometric.py:13-73,228-252, unidepth/utils/sht.py:833.  GEMM-shaped V1 work (every Linear, the stem /
 * downsample convolutions as im2col GEMMs, 1x1 and 3x3 convolutions, the 8x64-head attention blocks) reuses
 * udb_gemm_f16 / udb_attention_f16 above.
 * ============================================================================================= */

/* V1 pre-processing + stem im2col (unidepthv1.py:49-63,298-317; convnext.py:371-383): uint8 / f32 NCHW -> (/255) ->
 * ImageNet normalise -> antialiased bilinear to (rh, rw) -> zero pad (pad_l, pad_t) into (net_h, net_w) -> f16 rows
 * [B*gh*gw, 64] of the 4x4 stride-4 patches (column c*16 + py*4 + px, 48 used; gh = (net_h-4)/4+1). */
typedef struct udb_v1_preprocess_t {
  const void* rgb;
  int32_t rgb_is_u8, scale255, normalize;
  int32_t B, H, W;
  int32_t rh, rw, pad_l, pad_t;
  int32_t net_h, net_w;
  void* patches;
} udb_v1_preprocess_t;
int udb_v1_preprocess(const udb_v1_preprocess_t* p, void* stream);
/* The same pre-processing for the DINOv2 ViT encoder (V1 with dinov2_vit*14): 14x14 stride-14 patch rows
 * [B*gh*gw, 640] f16 (column c*196 + py*14 + px, 588 used, the rest zero; gh = net_h/14), the operand layout of the
 * patch-embedding GEMM. */
int udb_v1_preprocess_vit(const udb_v1_preprocess_t* p, void* stream);
/* ViT tap after one encoder block (unidepthv1.py:322-326, decoder.py:371-374).  x: f32 residual stream [B, T, D] (row 0 =
 * cls).  dst [B, T-1, D] f16: f16(x[b,1+n,:] + x[b,0,:]) when `first`, else the element-wise max of dst and that (the
 * running max over a block range).  cls (may be NULL): x[b,0,:] copied to [B, D] f32.  D % 8 == 0, 16-byte aligned. */
int udb_vit_tap_f16(const float* x, void* dst, float* cls, int32_t B, int32_t T, int32_t D, int32_t first, void* stream);

/* LayerNorm over the last dim for widths that are multiples of 64 up to 1536 (ConvNeXt channel LayerNorm / LayerNorm2d,
 * convnext.py:214,252-263; decoder LayerNorms).  in row r at in + r*ld_in (+ add[(r % add_mod)*dim ..] when add != NULL:
 * "tokens + positional embedding", decoder.py:92-94,224).  s2d_w > 0: rows are the pixels of [B, s2d_h, s2d_w] maps and
 * pixel (y,x) is written to row (b, y/2, x/2), columns ((y&1)*2+(x&1))*dim.. of the k2 s2 downsample's im2col matrix
 * [B*(s2d_h/2)*(s2d_w/2), ld_out] (a trailing odd row / column is dropped, as the strided convolution drops it). */
typedef struct udb_layernorm_any_t {
  const void* in;
  int32_t in_f32;
  void* out;
  int32_t out_f32;
  const float* weight;
  const float* bias;
  int64_t rows;
  int32_t dim;
  int64_t ld_in, ld_out;
  float eps;
  const float* add;
  int64_t add_mod;
  int32_t s2d_h, s2d_w;
} udb_layernorm_any_t;
int udb_layernorm_any(const udb_layernorm_any_t* p, void* stream);

/* Depthwise 7x7, zero padding 3 (convnext.py:208-211 conv_dw; layers/convnext.py:16-24 dwconv): x f16 NHWC [B,H,W,C],
 * w f32 [49, C] (tap-major), bias f32 [C] -> y f16 NHWC.  C % 64 == 0. */
int udb_dwconv7_nhwc_f16(const void* x, const float* w, const float* bias, void* y, int32_t B, int32_t H, int32_t W,
                         int32_t C, void* stream);

/* dst = first ? src : max(dst, src) element-wise over n f16 values (decoder.py:371-374 max_stack over a stage's blocks). */
int udb_max_accum_f16(const void* src, void* dst, int64_t n, int32_t first, void* stream);

/* Mean over the HW pixels of an f32 NHWC map -> [B, C] (ConvNeXt "cls tokens", convnext.py:471). */
int udb_spatial_mean_f32(const float* x, float* out, int32_t B, int32_t HW, int32_t C, void* stream);

/* F.interpolate(bilinear, align_corners=False, antialias=True) of an f16 NHWC map (flat_interpolate, geometric.py:228-252). */
int udb_aa_resize_nhwc_f16(const void* in, void* out, int32_t B, int32_t H, int32_t W, int32_t C, int32_t oh, int32_t ow,
                           void* stream);

/* Ray embedding of one decoder level (decoder.py:203-220): analytic unit rays of K (intr4 = fx,fy,cx,cy per image, network
 * resolution) antialias-averaged per token, re-normalised, 81 real spherical harmonics (sht.py:833, index l*(l+1)+m),
 * then the projection MLP's input LayerNorm (ln_w / ln_b [81], eps 1e-5).  out f16 [B*gh*gw, 128], columns >= 81 zero.
 * sh_k[l*9+m] = K_l^m (times sqrt(2) for m > 0). */
typedef struct udb_v1_rays_t {
  const float* intr4;
  int32_t B, net_h, net_w, gh, gw;
  const float* ln_w;
  const float* ln_b;
  void* out;
  float sh_k[81];
} udb_v1_rays_t;
int udb_v1_rays_sh81(const udb_v1_rays_t* p, void* stream);

/* Camera head tail (decoder.py:96-106,326-331; unidepthv1.py:56-62,88-91,354-356).  x4 [B,4] (may be NULL with
 * skip_camera) -> intr4_rays [B,4]: K the decoder's rays use (prediction, or the pre-processed GT K); k_out [B,3,3]: the
 * intrinsics returned to the caller; k4_points [B,4]: K of the final back-projection. */
int udb_v1_camera_intrinsics(const float* x4, const float* gt_k, int32_t B, int32_t net_h, int32_t net_w, float ratio,
                             int32_t pad_l, int32_t pad_t, int32_t skip_camera, float* intr4_rays, float* k_out,
                             float* k4_points, void* stream);

/* Single-head cross attention with a handful of queries (camera head `aggregate`, decoder.py:95): q f32 [B*nq, D]
 * (+ q_pos [nq, D] when not NULL: the learned latents_pos, layers/attention.py:129-131; then scaled by `scale`),
 * kv f16 [B*nk, 2D] = (k | v), out f32 [B*nq, D].  nq <= 4, D % 256 == 0; scratch: B*16*nq*(D+2) floats (the keys are split
 * over 16 blocks per image, partial results are merged by a second kernel). */
int udb_cross_attn_small(const float* q, const float* q_pos, const void* kv, float* out, float* scratch, int32_t B, int32_t nq,
                         int32_t nk, int32_t D, float scale, void* stream);

/* p[r, j] = softmax_j(scale * s[r, j]) over j < n_valid, f32 [rows, ld_in] -> f16 [rows, ld_out], columns >= n_valid zero
 * (the P operand of the dense single-head attentions aggregate_16 / prompt_camera, decoder.py:231-236). */
int udb_softmax_rows(const float* s, void* p, int64_t rows, int32_t n_valid, int32_t ld_in, int32_t ld_out, float scale,
                     void* stream);

/* out = a + b (f32; out and/or an f16 copy), n % 4 == 0 (decoder.py:246-252 `latents + rays_embedding`). */
int udb_add_f32(const float* a, const float* b, float* out, void* out_f16, int64_t n, void* stream);

/* f32 [groups*rows_per_group, D] -> f16 rows (g*dst_group_stride + dst_row0 + r) of dst (decoder.py:94 torch.cat). */
int udb_copy_rows_f32_to_f16(const float* src, void* dst, int32_t groups, int32_t rows_per_group, int32_t D,
                             int64_t dst_group_stride, int64_t dst_row0, void* stream);

/* exp(clamp(conv3x3(x; w [9, C], bias), -10, 10)) with one output channel, zero padding: x f16 NHWC -> f32 [B,H,W]
 * (decoder.py:253,268,283,292-294 out8 / out4 / out2). */
int udb_conv3x3_c1_exp(const void* x, const float* w, float bias, float* out, int32_t B, int32_t H, int32_t W, int32_t C,
                       void* stream);

/* Nystrom attention pieces (layers/nystrom_attention.py:22-84 -> xformers NystromAttention(num_landmarks=128); restated
 * algorithm and its "parity unpinned" status: oracle/unidepth_v1_oracle.py).  64-wide heads.
 * landmarks: segment means of q (qbuf [B*n, ldq]) and k (kvbuf [B*n, ldkv]) -> f16 [B*128, 2*heads*64] = (ql | kl).
 * k2_pinv:   kernel_2 = softmax(ql kl^T / 8) -> k2 [B*heads,128,128] f32; z = its Newton-Schulz pseudo-inverse
 *            (`iters` steps, tmp = 3 * B*heads*128*128 floats).
 * zk3:       out[(b, lm), h*64+d] = sum_j z[b,h][lm][j] * k3[(b, j), h*64+d]   (f16 in / out). */
int udb_nystrom_landmarks(const void* q, int32_t ldq, const void* kv, int32_t ldkv, void* out, int32_t B, int32_t n,
                          int32_t heads, void* stream);
int udb_nystrom_k2_pinv(const void* landmarks, float* k2, float* z, float* tmp, int32_t B, int32_t heads, int32_t iters,
                        void* stream);
int udb_nystrom_zk3(const float* z, const void* k3, int32_t ldk3, void* out, int32_t ldo, int32_t B, int32_t heads, void* stream);

/* V1 post-processing (unidepthv1.py:66-94,352-366).  mean_maps: the three exp'ed maps (gh*2, gh*4, gh*8 grids) antialias-
 * resized to the network shape and averaged.  postprocess: crop the paddings, antialias-resize to (H, W) -> depth; points =
 * spherical_zbuffer_to_euclidean(theta, phi, z) with the angles of the unit ray of k4 (fx,fy,cx,cy) through each pixel. */
int udb_v1_mean_maps(const float* o8, const float* o4, const float* o2, float* mean, int32_t B, int32_t gh, int32_t gw,
                     int32_t net_h, int32_t net_w, void* stream);
typedef struct udb_v1_postprocess_t {
  const float* mean;
  const float* k4;
  int32_t B, net_h, net_w, pad_l, pad_r, pad_t, pad_b, H, W;
  float* out_depth;
  float* out_points;
} udb_v1_postprocess_t;
int udb_v1_postprocess(const udb_v1_postprocess_t* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Output assembly (unidepthv2.py:80-89, 311-339, 375-377; unidepthv2/decoder.py:456-462):
 * radius/confidence f32 [B,net_h,net_w] (already exp'ed), rays from intr4 (or rays_in) ->
 * points = rays*radius -> bilinear (align_corners=False) to (padded_h, padded_w) -> crop pads ->
 * confidence[B,1,H,W], radius[B,1,H,W]=|points|, depth[B,1,H,W]=points.z, points[B,3,H,W],
 * rays[B,3,H,W] renormalised.  All f32.
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_postprocess_t {
  const float* radius;
  const float* confidence;
  const float* intr4;
  const float* rays_in; /* optional [B, net_h*net_w, 3] */
  int32_t B, net_h, net_w, padded_h, padded_w, pad_l, pad_t, H, W;
  float* out_confidence;
  float* out_radius;
  float* out_depth;
  float* out_points;
  float* out_rays;
} udb_postprocess_t;
int udb_postprocess(const udb_postprocess_t* p, void* stream);

/* ======================================================================================
 * Whole-path engine: one handle = one UniDepthV2 model on one device.
 *
 * Replaces the body of `UniDepthV2.infer` (unidepth/models/unidepthv2/unidepthv2.py:239-339:
 * pre-process -> `encode_decode` :341-377 -> `_postprocess` :80-108) as ONE call that only enqueues
 * kernels on the caller's stream: no allocation, no host<->device copy, no synchronisation, so the
 * call is CUDA-graph capturable.  The caller (the Python boundary class, or any C program) owns all
 * memory: packed weights, the workspace and the seven output tensors.
 *
 * Life cycle:   udb_create -> udb_set_weight / udb_set_scalar (once per packed tensor)
 *               -> udb_workspace_bytes(B,H,W,level)  [per new input shape; also prepares the
 *                  shape-dependent tables: resized position embedding, ray-embedding frequencies]
 *               -> udb_infer_v2 (any number of times) -> udb_destroy.
 * A handle is not thread-safe (neither is a reference model instance: `infer` mutates module state,
 * decoder.py:436,447-448).  All functions return 0 on success, non-zero + udb_last_error() otherwise.
 * ====================================================================================== */
typedef struct udb_engine udb_engine;

enum { UDB_DT_F16 = 0, UDB_DT_F32 = 1 };

typedef struct udb_config_t {
  /* DINOv2 encoder (unidepth/models/backbones/dinov2.py:388-427, encoder.py:139-193) */
  int32_t embed_dim, depth, enc_heads;
  int32_t taps[4];      /* 1-based indices of the four block outputs consumed (unidepthv2.py:365-372) */
  int32_t pos_grid;     /* side of the stored position-embedding grid (37) */
  /* decoder (unidepth/models/unidepthv2/decoder.py:470-524) */
  int32_t hidden, dec_heads, expansion, out_dim;
  int32_t n_stages;     /* len(depths) */
  int32_t dec_depths[4];
  /* data.augmentations.shape_constraints of the model config (unidepthv2.py:247-262) */
  double ratio_min, ratio_max;
  double pixels_min, pixels_max;
} udb_config_t;

int udb_create(const udb_config_t* cfg, udb_engine** out);
void udb_destroy(udb_engine* e);

/* Register one PACKED tensor (device pointer, borrowed for the life of the handle) under the engine's
 * own name; the packing (f16 operand layouts, folded LayerNorm->Linear heads, zero-padded narrow
 * heads) is described in DESIGN.md and done once per checkpoint by the boundary class from the
 * reference's state_dict (SURVEY.md 8b).  dtype: UDB_DT_*. */
int udb_set_weight(udb_engine* e, const char* name, const void* dev_ptr, const int64_t* shape, int32_t ndim,
                   int32_t dtype);
/* Host scalars of the packed model (the two 1x1 head biases and their additive constants). */
int udb_set_scalar(udb_engine* e, const char* name, double value);

/* Geometry of one call, same arithmetic as get_paddings / get_resize_factor (unidepthv2.py:36-77). */
typedef struct udb_geometry_t {
  int32_t pad_l, pad_r, pad_t, pad_b;
  int32_t padded_h, padded_w;
  int32_t net_h, net_w;   /* network input, multiples of 14 */
  int32_t gh, gw;         /* patch grid */
  double factor;
} udb_geometry_t;
/* resolution_level: 0..9, -1 = attribute unset (default pixel bounds), or UDB_LEVEL_NETWORK_ONLY: the input
 * already is the network input (normalised float tensor, H and W multiples of 14): identity geometry, the
 * outputs are the network's own (the reference's `encode_decode` as used by `forward_test`,
 * unidepthv2.py:134-160, and by the ONNX wrappers, export.py:27-45). */
#define UDB_LEVEL_NETWORK_ONLY (-2)
int udb_geometry(const udb_engine* e, int32_t H, int32_t W, int32_t resolution_level, udb_geometry_t* out);

/* Bytes of scratch udb_infer_v2 needs for this shape; also prepares the per-shape tables (may
 * allocate and launch on the default stream: call it outside graph capture). 0 = error. */
size_t udb_workspace_bytes(udb_engine* e, int32_t B, int32_t H, int32_t W, int32_t resolution_level);
/* The same number from a dry run of the schedule alone: walks every stage with the registered operands, checks their
 * names and shapes, sizes the bump allocator -- and touches no device (no table is prepared, nothing is recorded), so it
 * also works on a machine without a GPU.  udb_infer_v2 still requires udb_workspace_bytes.  0 = error. */
size_t udb_schedule_bytes(udb_engine* e, int32_t B, int32_t H, int32_t W, int32_t resolution_level);

typedef struct udb_infer_args_t {
  const void* rgb;            /* [B,3,H,W] uint8 or float32 (0..255 when normalize) */
  int32_t rgb_is_u8, normalize;
  int32_t B, H, W;
  int32_t resolution_level;   /* 0..9 or -1 */
  const float* camera_k;      /* optional [B,3,3] pinhole K in input-image pixels (infer(camera=K),
                                 unidepthv2.py:267-303): rays come from it, intrinsics stay predicted */
  const float* camera_rays;   /* optional [B, net_h*net_w, 3] unit rays at network-input resolution produced by the
                                 caller's camera model (infer(camera=<Camera object>): camera.crop / resize /
                                 get_rays, unidepthv2.py:299-303,361-362; decoder.py:400); overrides camera_k */
  const float* ray_scales;    /* optional [hidden/2] frequency table (positional_embedding.py:231-233);
                                 NULL = the engine's own table */
  void* workspace;
  size_t workspace_bytes;
  /* outputs, float32, caller-allocated (keys of the dict returned by infer, unidepthv2.py:331-339) */
  float* confidence;          /* [B,1,H,W] */
  float* intrinsics;          /* [B,3,3]   */
  float* radius;              /* [B,1,H,W] */
  float* depth;               /* [B,1,H,W] */
  float* points;              /* [B,3,H,W] */
  float* rays;                /* [B,3,H,W] */
  float* depth_features;      /* [B,gh,gw,hidden] channel-last (the reference returns the same values
                                 as [B,hidden,gh,gw]; the boundary class returns a permuted view) */
} udb_infer_args_t;

int udb_infer_v2(udb_engine* e, const udb_infer_args_t* a, void* stream);

/* ---------------------------------------------------------------------------------------------
 * UniDepthV1 engine: the whole `UniDepthV1.infer` path (ConvNeXt encoder) as one call (SURVEY.md section 8b
 * `udb_infer_v1`; reference unidepth/models/unidepthv1/unidepthv1.py:288-373).  Same contract as the V2 engine: the
 * caller owns packed weights (names listed in unidepth_b200/unidepthv1.py::_pack), workspace and outputs; nothing is
 * allocated, copied or synchronised inside udb_infer_v1.
 * ------------------------------------------------------------------------------------------- */
typedef struct udb_engine_v1 udb_engine_v1;

typedef struct udb_v1_config_t {
  int32_t depths[4];      /* ConvNeXt blocks per stage (convnext_large: 3,3,27,3) */
  int32_t dims[4];        /* stage widths (192,384,768,1536) */
  int32_t hidden, heads, expansion;
  int32_t dec_depths[3];  /* attention blocks at 1/16, Nystrom blocks at 1/8 and 1/4 (config pixel_decoder.depths) */
  int32_t net_h, net_w;   /* fixed network input (config data.image_shape: 462 x 616) */
} udb_v1_config_t;

int udb_v1_create(const udb_v1_config_t* cfg, udb_engine_v1** out);
/* UniDepthV1 with a DINOv2 ViT encoder (dinov2_vit*14, e.g. config_v1_vitl14.json): cfg->depths hold the lengths of
 * the four block ranges the decoder max-stacks (ViT-L with output_idx 5,12,18,24: 5,7,6,6), cfg->dims the embedding
 * width four times, enc_heads the encoder's heads (64-wide).  The network shape must be a multiple of 14.  Encoder
 * operands: patch_w [D, 640] f16 (588 used), patch_b, cls [D], pos [1 + gh*gw, D] f32 (the position table already
 * resampled to the network grid), blocks.<i>.{n1w,n1b,qkv_w,qkv_b,proj_w,proj_b,ls1,n2w,n2b,fc1_w,fc1_b,fc2_w,fc2_b,ls2}
 * as in the V2 engine's default mode; the decoder's are the ConvNeXt model's. */
int udb_v1_create_vit(const udb_v1_config_t* cfg, int32_t enc_heads, udb_engine_v1** out);
void udb_v1_destroy(udb_engine_v1* e);
int udb_v1_set_weight(udb_engine_v1* e, const char* name, const void* dev_ptr, const int64_t* shape, int32_t ndim,
                      int32_t dtype);
int udb_v1_set_scalar(udb_engine_v1* e, const char* name, double value);
/* Shape arithmetic of one V1 call, the engine's own copy of `_shapes` / `_paddings` (unidepthv1.py:30-46): the image is resized
 * by `ratio` to (resized_h, resized_w) -- the larger side-ratio that still fits the fixed network input -- and zero-padded
 * (pad_* >= 0 here; Python floor division kept for the general case) to net_h x net_w. */
typedef struct udb_v1_geometry_t {
  int32_t resized_h, resized_w;
  int32_t pad_l, pad_r, pad_t, pad_b;
  double ratio;
} udb_v1_geometry_t;
int udb_v1_geometry(int32_t H, int32_t W, int32_t net_h, int32_t net_w, udb_v1_geometry_t* out);
/* bytes of workspace udb_infer_v1 needs for this shape (0 + udb_last_error on failure); must be called once per
 * (B, H, W) after the weights are registered and outside stream capture */
size_t udb_v1_workspace_bytes(udb_engine_v1* e, int32_t B, int32_t H, int32_t W);

typedef struct udb_infer_v1_args_t {
  const void* rgb;        /* [B,3,H,W] uint8 or float32 */
  int32_t rgb_is_u8;
  int32_t scale255;       /* divide by 255 first (uint8, or float data with max > 5: unidepthv1.py:301-302) */
  int32_t normalize;      /* ImageNet mean / std (data in [0,1] after the optional /255: unidepthv1.py:303-308) */
  int32_t B, H, W;
  const float* intrinsics; /* optional GT pinhole K [B,3,3] (original image frame) */
  int32_t skip_camera;     /* with intrinsics: do not run the camera head, return the GT K (unidepthv1.py:336) */
  void* workspace;
  size_t workspace_bytes;
  float* out_intrinsics;  /* [B,3,3] */
  float* out_points;      /* [B,3,H,W] */
  float* out_depth;       /* [B,1,H,W] */
} udb_infer_v1_args_t;

int udb_infer_v1(udb_engine_v1* e, const udb_infer_v1_args_t* a, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Peer-memory plumbing of the multi-GPU output gather (one process per GPU on one node; SURVEY.md section 8e).
 * alloc: device buffer (zero-filled) + its 64-byte CUDA IPC handle, to be exchanged out of band (torch.distributed);
 * open: map a peer's buffer; barrier: device-side barrier over flags in peer memory (flag arrays of `world` uint32,
 * peer_flags_dev = device array of the ranks' flag-array pointers as mapped HERE; epochs only grow; a missing peer sets
 * *timeout_flag_dev instead of hanging); copy: copy-engine device-to-device copy (no SM involved).
 * ------------------------------------------------------------------------------------------- */
int udb_p2p_alloc(size_t bytes, void** dev_ptr, void* handle64);
int udb_p2p_open(const void* handle64, void** peer_ptr);
int udb_p2p_close(void* peer_ptr);
int udb_p2p_free(void* dev_ptr);
int udb_p2p_barrier(void* const* peer_flags_dev, void* my_flags, int32_t rank, int32_t world, uint32_t epoch,
                    int32_t* timeout_flag_dev, void* stream);
int udb_p2p_copy(void* dst, const void* src, size_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UDB_H_ */
