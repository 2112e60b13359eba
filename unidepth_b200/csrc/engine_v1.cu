// Whole-path engine for UniDepthV1.infer with the ConvNeXt encoder (BASELINE config 4) or a DINOv2 ViT encoder, behind
// udb_v1_create / udb_v1_create_vit / udb_v1_set_weight / udb_v1_workspace_bytes / udb_infer_v1 (include/udb.h).  Host-side schedule only: it enqueues the
// kernels of this library on the caller's stream over a bump-allocated workspace (no allocation, copy or sync inside
// udb_infer_v1, so the call is graph-capturable).  Reference call stack it replaces:
//   UniDepthV1.infer                 unidepth/models/unidepthv1/unidepthv1.py:288-373 (_shapes/_paddings/_preprocess/_postprocess :30-94)
//     pixel_encoder = ConvNeXt       unidepth/models/backbones/convnext.py:459-471 (stem :371-383, stage :289-298, block :208-223)
//                   or DINOv2        unidepth/models/backbones/dinov2.py:306-347 (all blocks, no final norm; + cls, unidepthv1.py:322-326)
//     pixel_decoder = Decoder        unidepth/models/unidepthv1/decoder.py:364-463 (run_camera :311-343, CameraHead :85-106,
//                                    DepthHead :195-300), layers/{attention,nystrom_attention,mlp,upsample,convnext}.py
#include <stdlib.h>

#include "engine_common.h"

struct udb_engine_v1 : udb::EngineBase {
  udb_v1_config_t cfg;
  int vit_heads = 0;                                  // > 0: DINOv2 ViT encoder (udb_v1_create_vit)
  std::unordered_map<std::string, size_t> ws_need;   // "B,H,W" -> bytes
};

namespace udb {

struct V1Geom {
  int rh, rw;                       // resized image inside the network frame
  double ratio;
  int pad_l, pad_r, pad_t, pad_b;
};

// unidepthv1.py:30-46 (Python float == C double; ceil(x - 0.5))
static V1Geom v1_geometry(int H, int W, int net_h, int net_w) {
  V1Geom g;
  const double in_ratio = static_cast<double>(W) / H, out_ratio = static_cast<double>(net_w) / net_h;
  g.ratio = out_ratio > in_ratio ? static_cast<double>(net_h) / H : static_cast<double>(net_w) / W;
  g.rh = static_cast<int>(ceil(H * g.ratio - 0.5));
  g.rw = static_cast<int>(ceil(W * g.ratio - 0.5));
  const int dh = net_h - g.rh, dw = net_w - g.rw;
  const auto fdiv2 = [](int v) { return v >= 0 ? v / 2 : -((-v + 1) / 2); };
  g.pad_t = fdiv2(dh); g.pad_b = dh - g.pad_t;
  g.pad_l = fdiv2(dw); g.pad_r = dw - g.pad_l;
  return g;
}

struct V1Ctx : Ctx {
  // Debug taps: with UDB_V1_DUMP=<dir> set (and the call NOT under stream capture) named intermediates are written as raw
  // files <dir>/<name>.bin after a stream sync; tests/tools compare them with the oracle's taps.  Off in normal operation.
  void tap(const char* name, const void* p, size_t bytes) {
    static const char* dir = getenv("UDB_V1_DUMP");
    if (!dir || dry || rc) return;
    cudaStreamSynchronize(static_cast<cudaStream_t>(st));
    std::vector<char> host(bytes);
    if (cudaMemcpy(host.data(), p, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return;
    const std::string path = std::string(dir) + "/" + name + ".bin";
    if (FILE* f = fopen(path.c_str(), "wb")) { fwrite(host.data(), 1, bytes, f); fclose(f); }
  }
  void ln_any(const void* in, int in_f32, void* out, int out_f32, const float* w, const float* b, long long rows, int dim, float eps,
              long long ld_out = 0, const float* add = nullptr, long long add_mod = 0, int s2d_h = 0, int s2d_w = 0) {
    if (dry || rc) return;
    udb_layernorm_any_t p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.in_f32 = in_f32; p.out = out; p.out_f32 = out_f32; p.weight = w; p.bias = b;
    p.rows = rows; p.dim = dim; p.ld_in = dim; p.ld_out = ld_out ? ld_out : dim; p.eps = eps;
    p.add = add; p.add_mod = add_mod; p.s2d_h = s2d_h; p.s2d_w = s2d_w;
    done(udb_layernorm_any(&p, st));
  }
  // LayerNorm to f16 for any decoder / encoder width: the V2 kernels where they apply (128-multiples up to 1024 from f32,
  // 64/128/256 from f16), the generic one otherwise
  void ln16(const void* in, int in_f32, void* out, const std::string& wn, const std::string& bn, long long rows, int dim, float eps) {
    const bool v2_ok = in_f32 ? (dim % 128 == 0 && dim <= 1024) : (dim == 64 || dim == 128 || dim == 256 || (dim % 128 == 0 && dim <= 1024));
    if (v2_ok) layernorm(in, in_f32, out, 0, F(wn), F(bn), static_cast<int>(rows), dim, eps);
    else ln_any(in, in_f32, out, 0, F(wn), F(bn), rows, dim, eps);
  }
  // MLP tail on the f32 residual stream x [rows, C]:  x += gamma * (W2 gelu(W1 LN(x) + b1) + b2)        (layers/mlp.py:9-35)
  void mlp_resid(const std::string& p, float* x, long long rows, int C, int mid, const float* gamma, __half* x16 = nullptr) {
    const size_t m = ar->mark();
    __half* hN = ar->h(rows * C);
    __half* md = ar->h(rows * mid);
    ln16(x, 1, hN, p + "nw", p + "nb", rows, C, 1e-5f);
    { G q{hN, H(p + "w1"), static_cast<int>(rows), mid, C}; q.bias = F(p + "b1"); q.act = UDB_ACT_GELU; q.out = md; gemm(q); }
    { G q{md, H(p + "w2"), static_cast<int>(rows), C, mid}; q.bias = F(p + "b2"); q.gamma = gamma; q.resid = x; q.resid_f32 = 1;
      q.out = x; q.out_f32 = 1; q.out2 = x16; q.out2_leaky = 0; gemm(q); }
    ar->release(m);
  }
  // ConvNeXt-style block on an NHWC map: x f32 (+ its f16 copy x16) [B,H,W,C] updated in place
  // (convnext.py:208-223 with eps 1e-6; layers/convnext.py:34-44 with eps 1e-5)
  void cvnxt_block(const std::string& p, float* x, __half* x16, int B, int Hh, int Ww, int C, float eps) {
    const size_t m = ar->mark();
    const long long rows = static_cast<long long>(B) * Hh * Ww;
    __half* y = ar->h(rows * C);
    __half* hN = ar->h(rows * C);
    __half* md = ar->h(rows * 4 * C);
    if (!dry && !rc) done(udb_dwconv7_nhwc_f16(x16, F(p + "dw_w"), F(p + "dw_b"), y, B, Hh, Ww, C, st));
    ln16(y, 0, hN, p + "ln_w", p + "ln_b", rows, C, eps);
    { G q{hN, H(p + "w1"), static_cast<int>(rows), 4 * C, C}; q.bias = F(p + "b1"); q.act = UDB_ACT_GELU; q.out = md; gemm(q); }
    { G q{md, H(p + "w2"), static_cast<int>(rows), C, 4 * C}; q.bias = F(p + "b2"); q.gamma = F(p + "gamma"); q.resid = x; q.resid_f32 = 1;
      q.out = x; q.out_f32 = 1; q.out2 = x16; q.out2_leaky = 0; gemm(q); }
    ar->release(m);
  }
  void attention_sp(const void* q, const void* k, const void* v, void* out, int B, int heads, int sq, int sk, int ldq, int ldk, int ldv, int ldo,
                    int q0, int k0, int v0) {
    attention(q, k, v, out, B, heads, sq, sk, ldq, ldk, ldv, ldo, q0, k0, v0, 0.125f);
  }
};

static inline long long rup(long long v, long long m) { return (v + m - 1) / m * m; }

// DINOv2 encoder of V1 (dinov2.py:306-347 with interpolate_offset 0.1, unidepthv1.py:322-326, decoder.py:371-379): 14x14
// patches -> patch GEMM + position table -> cls row -> all blocks; after each block the (x + cls) map is max-stacked into
// its range's level and the last four blocks' cls rows are kept (clsbuf[k]: block last - k).
static void vit_encoder_v1(V1Ctx& c, const udb_infer_v1_args_t& a, const V1Geom& g, int vit_heads, int gh, int gw, __half* const* levels,
                           float* const* clsbuf) {
  const udb_v1_config_t& cf = static_cast<udb_engine_v1*>(c.e)->cfg;
  Arena& ar = *c.ar;
  const int B = a.B, N = gh * gw, T = N + 1, D = cf.dims[0];
  const size_t BN = static_cast<size_t>(B) * N, BT = static_cast<size_t>(B) * T;
  __half* patches = ar.h(BN * 640);
  if (!c.dry) {
    udb_v1_preprocess_t p;
    memset(&p, 0, sizeof(p));
    p.rgb = a.rgb; p.rgb_is_u8 = a.rgb_is_u8; p.scale255 = a.scale255; p.normalize = a.normalize; p.B = B; p.H = a.H; p.W = a.W;
    p.rh = g.rh; p.rw = g.rw; p.pad_l = g.pad_l; p.pad_t = g.pad_t; p.net_h = cf.net_h; p.net_w = cf.net_w; p.patches = patches;
    c.done(udb_v1_preprocess_vit(&p, c.st));
  }
  c.expect2("pos", T, D);                    // the position table is packed for this network grid
  float* x = ar.f(BT * D);
  {
    Ctx::G q{patches, c.H("patch_w"), static_cast<int>(BN), D, 640};
    q.bias = c.F("patch_b"); q.resid = c.F("pos"); q.resid_f32 = 1; q.ldr = D; q.out = x; q.out_f32 = 1;
    q.rows_per_group = N; q.group_stride = T; q.row_offset = 1; q.resid_mod = N; q.resid_row_offset = 1;
    c.expect2("patch_w", D, 640);
    c.gemm(q);
    const float* cls = c.F("cls");           // looked up in the dry run too, so a missing one is reported there
    if (!c.dry && !c.rc) c.done(udb_set_cls_rows(x, cls, c.F("pos"), B, T, D, c.st));
  }
  const VitScratch vs{ar.h(BT * D), ar.h(BT * 3 * D), ar.h(BT * D), ar.h(BT * 4 * D), nullptr, nullptr, 0, 0};
  int total = 0;
  for (int l = 0; l < 4; ++l) total += cf.depths[l];
  for (int l = 0, i = 0; l < 4; ++l)
    for (int j = 0; j < cf.depths[l]; ++j, ++i) {
      vit_block(c, idx("blocks.%d.", i), x, B, T, D, vit_heads, false, false, vs);
      const int from_end = total - 1 - i;
      if (!c.dry && !c.rc) c.done(udb_vit_tap_f16(x, levels[l], from_end < 4 ? clsbuf[from_end] : nullptr, B, T, D, j == 0, c.st));
      if (i == 0) c.tap("enc_block0", x, sizeof(float) * BT * D);
    }
  c.tap("enc_last", x, sizeof(float) * BT * D);
}

// Single-head (head dim = D) attention block with a separate context (decoder.py:225-236 aggregate_16 / prompt_camera),
// computed densely: S = q k^T (GEMM) -> row softmax -> P v (GEMM with v^T as the K-major operand).
static void dense_attn_block(V1Ctx& c, const std::string& p, float* x, int B, int nq, int D, const void* ctx, int ctx_f32, int nk,
                             const float* pos_ctx) {
  Arena& ar = *c.ar;
  const size_t m = ar.mark();
  const long long Rq = static_cast<long long>(B) * nq, Rk = static_cast<long long>(B) * nk;
  const int kp = static_cast<int>(rup(nk, 64));
  __half* xn = ar.h(Rq * D);
  __half* cn = ar.h((Rk + 64) * D);
  c.ln16(x, 1, xn, p + "nxw", p + "nxb", Rq, D, 1e-5f);
  c.ln16(ctx, ctx_f32, cn, p + "ncw", p + "ncb", Rk, D, 1e-5f);
  if (!c.dry && !c.rc) cudaMemsetAsync(cn + Rk * D, 0, sizeof(__half) * 64 * D, static_cast<cudaStream_t>(c.st));
  __half* q = ar.h(Rq * D);
  { Ctx::G g{xn, c.H(p + "q_w"), static_cast<int>(Rq), D, D}; g.bias = c.F(p + "q_b"); g.out = q; c.gemm(g); }
  __half* k = ar.h(static_cast<long long>(B) * kp * D);
  if (!c.dry && !c.rc) cudaMemsetAsync(k, 0, sizeof(__half) * B * kp * D, static_cast<cudaStream_t>(c.st));
  { Ctx::G g{cn, c.H(p + "k_w"), static_cast<int>(Rk), D, D}; g.bias = c.F(p + "k_b"); g.out = k;
    g.rows_per_group = nk; g.group_stride = kp; g.row_offset = 0;
    if (pos_ctx) { g.resid = pos_ctx; g.resid_f32 = 1; g.ldr = D; g.resid_mod = nk; g.resid_row_offset = 0; }
    c.gemm(g); }
  __half* vt = ar.h(static_cast<long long>(B) * D * kp);
  float* S = ar.f(static_cast<long long>(nq) * kp);
  __half* P = ar.h(static_cast<long long>(nq) * kp);
  __half* o = ar.h(Rq * D);
  const float scale = 1.0f / sqrtf(static_cast<float>(D));
  for (int b = 0; b < B; ++b) {
    // v^T [D, kp] = W_v . ctx_b^T  (the value bias is added after P v: softmax rows sum to 1)
    { Ctx::G g{c.H(p + "v_w"), cn + static_cast<long long>(b) * nk * D, D, kp, D}; g.out = vt + static_cast<long long>(b) * D * kp; c.gemm(g); }
    { Ctx::G g{q + static_cast<long long>(b) * nq * D, k + static_cast<long long>(b) * kp * D, nq, kp, D}; g.out = S; g.out_f32 = 1; c.gemm(g); }
    if (!c.dry && !c.rc) c.done(udb_softmax_rows(S, P, nq, nk, kp, kp, scale, c.st));
    { Ctx::G g{P, vt + static_cast<long long>(b) * D * kp, nq, D, kp}; g.bias = c.F(p + "v_b"); g.out = o + static_cast<long long>(b) * nq * D; c.gemm(g); }
  }
  { Ctx::G g{o, c.H(p + "out_w"), static_cast<int>(Rq), D, D}; g.bias = c.F(p + "out_b"); g.gamma = c.F(p + "ls1"); g.resid = x; g.resid_f32 = 1;
    g.out = x; g.out_f32 = 1; c.gemm(g); }
  ar.release(m);
  c.mlp_resid(p + "m", x, Rq, D, 4 * D, c.F(p + "ls2"));
}

// Multi-head self-attention block with 64-wide heads and a positional term added to q (decoder.py:239-241,256-258,271-273):
// exact attention (AttentionBlock) or the Nystrom approximation with 128 landmarks (NystromBlock).
static void mh_attn_block(V1Ctx& c, const std::string& p, float* x, int B, int n, int C, int heads, const float* pos, bool nystrom) {
  Arena& ar = *c.ar;
  const size_t m = ar.mark();
  const long long R = static_cast<long long>(B) * n;
  __half* xn = ar.h(R * C);
  __half* cn = ar.h(R * C);
  c.ln16(x, 1, xn, p + "nxw", p + "nxb", R, C, 1e-5f);
  c.ln16(x, 1, cn, p + "ncw", p + "ncb", R, C, 1e-5f);
  __half* q = ar.h(R * C);
  { Ctx::G g{xn, c.H(p + "q_w"), static_cast<int>(R), C, C}; g.bias = c.F(p + "q_b"); g.resid = pos; g.resid_f32 = 1; g.out = q; c.gemm(g); }
  __half* kv = ar.h(R * 2 * C);
  { Ctx::G g{cn, c.H(p + "kv_w"), static_cast<int>(R), 2 * C, C}; g.bias = c.F(p + "kv_b"); g.out = kv; c.gemm(g); }
  __half* o = ar.h(R * C);
  if (!nystrom) {
    c.attention_sp(q, kv, kv, o, B, heads, n, n, C, 2 * C, 2 * C, C, 0, 0, C);
  } else {
    const long long L = static_cast<long long>(B) * 128, mm = static_cast<long long>(B) * heads * 128 * 128;
    __half* lm = ar.h(L * 2 * C);          // (q landmarks | k landmarks)
    float* k2 = ar.f(mm);
    float* z = ar.f(mm);
    float* tmp = ar.f(3 * mm);
    __half* k3 = ar.h(L * C);
    __half* w2 = ar.h(L * C);
    if (!c.dry && !c.rc) c.done(udb_nystrom_landmarks(q, C, kv, 2 * C, lm, B, n, heads, c.st));
    if (!c.dry && !c.rc) c.done(udb_nystrom_k2_pinv(lm, k2, z, tmp, B, heads, 6, c.st));
    c.attention_sp(lm, kv, kv, k3, B, heads, 128, n, 2 * C, 2 * C, 2 * C, C, 0, 0, C);        // softmax(ql k^T) v
    if (!c.dry && !c.rc) c.done(udb_nystrom_zk3(z, k3, C, w2, C, B, heads, c.st));             // pinv . kernel_3
    c.attention_sp(q, lm, w2, o, B, heads, n, 128, C, 2 * C, C, C, 0, C, 0);                  // softmax(q kl^T) (pinv kernel_3)
  }
  { Ctx::G g{o, c.H(p + "out_w"), static_cast<int>(R), C, C}; g.bias = c.F(p + "out_b"); g.gamma = c.F(p + "ls1"); g.resid = x; g.resid_f32 = 1;
    g.out = x; g.out_f32 = 1; c.gemm(g); }
  ar.release(m);
  c.mlp_resid(p + "m", x, R, C, 4 * C, c.F(p + "ls2"));
}

// ConvUpsample (layers/upsample.py:13-45): (lat + emb) -> 2 CvnxtBlocks -> conv1x1 C->C/2 -> x2 bilinear (align_corners=True)
// -> conv3x3 (zero pad).  Returns the next level's f32 tokens and their f16 copy (allocated before the scratch mark).
static void conv_upsample(V1Ctx& c, const std::string& p, const float* lat, const float* emb, int B, int h, int w, int C, float* next,
                          __half* next16) {
  Arena& ar = *c.ar;
  const size_t m = ar.mark();
  const long long R = static_cast<long long>(B) * h * w;
  float* xs = ar.f(R * C);
  __half* xs16 = ar.h(R * C);
  if (!c.dry && !c.rc) c.done(udb_add_f32(lat, emb, xs, xs16, R * C, c.st));
  for (int j = 0; j < 2; ++j) c.cvnxt_block(p + (j ? "c1." : "c0."), xs, xs16, B, h, w, C, 1e-5f);
  const int C2 = C / 2;
  __half* u = ar.h(R * C2);
  { Ctx::G g{xs16, c.H(p + "up_w"), static_cast<int>(R), C2, C}; g.bias = c.F(p + "up_b"); g.out = u; c.gemm(g); }
  __half* up = ar.h(R * 4 * C2);
  if (!c.dry && !c.rc) c.done(udb_resize_ac_pad_nhwc_f16(u, up, B, h, w, C2, 2 * h, 2 * w, 0, c.st));
  c.expect2(p + "conv_w", C2, 9 * C2);
  c.conv3x3(up, B, 2 * h, 2 * w, C2, c.H(p + "conv_w"), C2, c.F(p + "conv_b"), UDB_ACT_NONE, nullptr, nullptr, 0, next, 1, next16, 0);
  ar.release(m);
}

static int run_v1(udb_engine_v1* e, const udb_infer_v1_args_t& a, Arena& ar, void* st) {
  const udb_v1_config_t& cf = e->cfg;
  V1Ctx c;
  c.e = e; c.ar = &ar; c.st = st; c.dry = ar.dry;
  const int B = a.B, net_h = cf.net_h, net_w = cf.net_w, hid = cf.hidden;
  const V1Geom g = v1_geometry(a.H, a.W, net_h, net_w);
  const bool vit = e->vit_heads > 0;
  int sh[4], sw[4];                 // level grids: the ConvNeXt pyramid, or the ViT patch grid four times
  sh[0] = vit ? net_h / 14 : (net_h - 4) / 4 + 1; sw[0] = vit ? net_w / 14 : (net_w - 4) / 4 + 1;
  for (int i = 1; i < 4; ++i) { sh[i] = vit ? sh[0] : sh[i - 1] / 2; sw[i] = vit ? sw[0] : sw[i - 1] / 2; }
  Stage stage;

  // ---- pre-processing + stem (convnext.py:371-383: conv k4 s4 as an im2col GEMM, then LayerNorm2d)
  stage.next("udb_v1:preprocess+stem");
  __half* levels[4];
  float* clsbuf[4];
  for (int i = 0; i < 4; ++i) levels[i] = ar.h(static_cast<size_t>(B) * sh[i] * sw[i] * cf.dims[i]);
  int total_blocks = 0;
  for (int i = 0; i < 4; ++i) total_blocks += cf.depths[i];
  // decoder.py:377-379: the cls tokens of the LAST FOUR BLOCKS, newest first
  int cls_dim[4];
  {
    int k = 0;
    for (int i = 3; i >= 0 && k < 4; --i)
      for (int j = cf.depths[i] - 1; j >= 0 && k < 4; --j) cls_dim[k++] = cf.dims[i];
    if (k != 4) { set_error("udb_infer_v1: the encoder needs at least four blocks"); return 1; }
  }
  for (int k = 0; k < 4; ++k) clsbuf[k] = ar.f(static_cast<size_t>(B) * cls_dim[k]);     // clsbuf[k]: block (last - k)
  if (vit) {
    stage.next("udb_v1:vit_encoder");
    const size_t enc_mark = ar.mark();
    vit_encoder_v1(c, a, g, e->vit_heads, sh[0], sw[0], levels, clsbuf);
    ar.release(enc_mark);
  } else {
    const size_t enc_mark = ar.mark();
    const long long n0 = static_cast<long long>(B) * sh[0] * sw[0];
    __half* patches = ar.h(n0 * 64);
    if (!c.dry) {
      udb_v1_preprocess_t p;
      memset(&p, 0, sizeof(p));
      p.rgb = a.rgb; p.rgb_is_u8 = a.rgb_is_u8; p.scale255 = a.scale255; p.normalize = a.normalize; p.B = B; p.H = a.H; p.W = a.W;
      p.rh = g.rh; p.rw = g.rw; p.pad_l = g.pad_l; p.pad_t = g.pad_t; p.net_h = net_h; p.net_w = net_w; p.patches = patches;
      c.done(udb_v1_preprocess(&p, st));
    }
    const int C0 = cf.dims[0];
    __half* y0 = ar.h(n0 * C0);
    { Ctx::G q{patches, c.H("stem_w"), static_cast<int>(n0), C0, 64}; q.bias = c.F("stem_b"); q.out = y0; c.gemm(q); }
    float* x = ar.f(n0 * C0);
    __half* x16 = ar.h(n0 * C0);
    c.ln_any(y0, 0, x, 1, c.F("stem_ln_w"), c.F("stem_ln_b"), n0, C0, 1e-6f);
    c.ln_any(y0, 0, x16, 0, c.F("stem_ln_w"), c.F("stem_ln_b"), n0, C0, 1e-6f);

    // ---- ConvNeXt stages (convnext.py:289-298); running max of each stage's block outputs (decoder.py:371-374)
    stage.next("udb_v1:convnext_stages");
    int blk = 0;
    for (int i = 0; i < 4; ++i) {
      const int C = cf.dims[i];
      const long long n = static_cast<long long>(B) * sh[i] * sw[i];
      if (i > 0) {
        const int Cp = cf.dims[i - 1];
        __half* A = ar.h(n * 4 * Cp);
        const std::string d = idx("ds%d.", i);
        c.ln_any(x, 1, A, 0, c.F(d + "ln_w"), c.F(d + "ln_b"), static_cast<long long>(B) * sh[i - 1] * sw[i - 1], Cp, 1e-6f, 4 * Cp, nullptr, 0,
                 sh[i - 1], sw[i - 1]);
        float* xn = ar.f(n * C);
        __half* xn16 = ar.h(n * C);
        c.expect2(d + "w", C, 4 * Cp);
        { Ctx::G q{A, c.H(d + "w"), static_cast<int>(n), C, 4 * Cp}; q.bias = c.F(d + "b"); q.out = xn; q.out_f32 = 1; q.out2 = xn16; q.out2_leaky = 0;
          c.gemm(q); }
        x = xn;
        x16 = xn16;
      }
      for (int j = 0; j < cf.depths[i]; ++j, ++blk) {
        c.cvnxt_block(idx2("s%d.b%d.", i, j), x, x16, B, sh[i], sw[i], C, 1e-6f);
        if (!c.dry && !c.rc) c.done(udb_max_accum_f16(x16, levels[i], n * C, j == 0, st));
        const int from_end = total_blocks - 1 - blk;
        if (from_end < 4 && !c.dry && !c.rc) c.done(udb_spatial_mean_f32(x, clsbuf[from_end], B, sh[i] * sw[i], C, st));
        if (blk == 0) c.tap("enc_block0", x, sizeof(float) * n * C);
      }
    }
    c.tap("enc_last", x, sizeof(float) * B * sh[3] * sw[3] * cf.dims[3]);
    ar.release(enc_mark);
  }

  // ---- decoder: common grid = second-smallest level (decoder.py:381-392; the ViT's one grid), adapters (:395-408)
  stage.next("udb_v1:adapters");
  const int hc = sh[2], wc = sw[2], nq = hc * wc;
  const long long Rq = static_cast<long long>(B) * nq;
  __half* featcat = ar.h(Rq * 4 * hid);                          // [B*nq, 4*hid]   (features_channels, decoder.py:224)
  __half* tokens = ar.h((Rq * 4 + 64) * hid);                    // [B, 4*nq, hid]  (features_tokens,   decoder.py:220)
  for (int l = 0; l < 4; ++l) {
    const size_t m = ar.mark();
    const int C = cf.dims[l];
    const __half* src = levels[l];
    if (sh[l] != hc || sw[l] != wc) {
      __half* r = ar.h(Rq * C);
      if (!c.dry && !c.rc) c.done(udb_aa_resize_nhwc_f16(levels[l], r, B, sh[l], sw[l], C, hc, wc, st));
      src = r;
    }
    __half* an = ar.h(Rq * C);
    const std::string ad = idx("adapt.%d.", l);
    c.ln16(src, 0, an, ad + "ln_w", ad + "ln_b", Rq, C, 1e-5f);
    { Ctx::G q{an, c.H(ad + "w"), static_cast<int>(Rq), hid, C}; q.bias = c.F(ad + "b"); q.act = UDB_ACT_GELU; q.out = tokens;
      q.rows_per_group = nq; q.group_stride = 4 * nq; q.row_offset = l * nq; c.gemm(q); }
    { Ctx::G q{an, c.H(ad + "w"), static_cast<int>(Rq), hid, C}; q.bias = c.F(ad + "b"); q.act = UDB_ACT_GELU; q.out = featcat + l * hid;
      q.ldc = 4 * hid; c.gemm(q); }
    ar.release(m);
  }
  c.tap("tokens", tokens, sizeof(__half) * Rq * 4 * hid);
  const float* tokens_pos = c.F("tokens_pos");                     // [4*nq, hid]: sine position + level embedding (decoder.py:410-433)
  {
    const Weight* tp = c.W("tokens_pos");
    if (!c.rc && (tp->shape[0] != 4LL * nq || tp->shape[1] != hid)) { set_error("engine_v1: tokens_pos must be [%d, %d]", 4 * nq, hid); return 1; }
  }

  // ---- camera head (decoder.py:311-343, 85-106), fp32 on the CUDA cores except the two context GEMMs
  stage.next("udb_v1:camera_head");
  float* intr4 = ar.f(static_cast<size_t>(B) * 4);
  float* k4_points = ar.f(static_cast<size_t>(B) * 4);
  const float* x4 = nullptr;
  if (!(a.skip_camera && a.intrinsics)) {
    const size_t m = ar.mark();
    const int R4 = B * 4;
    float* toks = ar.f(static_cast<size_t>(R4) * hid);
    for (int i = 0; i < 4; ++i) {
      const std::string tk = idx("tok.%d.", i);
      float* t = ar.f(static_cast<size_t>(B) * cls_dim[i]);
      c.ln_any(clsbuf[i], 1, t, 1, c.F(tk + "ln_w"), c.F(tk + "ln_b"), B, cls_dim[i], 1e-5f);
      c.small_linear(t, B, cls_dim[i], c.F(tk + "w"), hid, c.F(tk + "b"), UDB_ACT_GELU, nullptr, nullptr, toks + i * hid, cls_dim[i], 4 * hid, 0);
    }
    // cls_project: LN -> Linear(hid -> hid/2) -> GELU -> Linear(hid/2 -> hid)
    float* cl = cam_mlp(c, "cam.cls", toks, R4, hid, hid / 2, hid, nullptr, nullptr);
    // context = in_features(features + pos) ++ cls tokens
    const long long Rc = static_cast<long long>(B) * (4 * nq + 4);
    __half* ctx = ar.h(Rc * hid);
    {
      const size_t m2 = ar.mark();
      __half* a1 = ar.h(Rq * 4 * hid);
      __half* m1 = ar.h(Rq * 4 * 2 * hid);
      c.ln_any(tokens, 0, a1, 0, c.F("cam.inf.nw"), c.F("cam.inf.nb"), Rq * 4, hid, 1e-5f, 0, tokens_pos, 4LL * nq);
      { Ctx::G q{a1, c.H("cam.inf.w1"), static_cast<int>(Rq * 4), 2 * hid, hid}; q.bias = c.F("cam.inf.b1"); q.act = UDB_ACT_GELU; q.out = m1; c.gemm(q); }
      { Ctx::G q{m1, c.H("cam.inf.w2"), static_cast<int>(Rq * 4), hid, 2 * hid}; q.bias = c.F("cam.inf.b2"); q.out = ctx;
        q.rows_per_group = 4 * nq; q.group_stride = 4 * nq + 4; q.row_offset = 0; c.gemm(q); }
      ar.release(m2);
    }
    if (!c.dry && !c.rc) c.done(udb_copy_rows_f32_to_f16(cl, ctx, B, 4, hid, 4LL * nq + 4, 4LL * nq, st));
    // aggregate: the 4 tokens attend to the context (single head of width hid, position term on q)
    float* t;
    {
      const std::string ag = "cam.agg.";
      float* xn = ar.f(static_cast<size_t>(R4) * hid);
      c.layernorm(cl, 1, xn, 1, c.F(ag + "nxw"), c.F(ag + "nxb"), R4, hid, 1e-5f);
      __half* cn = ar.h(Rc * hid);
      c.ln16(ctx, 0, cn, ag + "ncw", ag + "ncb", Rc, hid, 1e-5f);
      __half* kv = ar.h(Rc * 2 * hid);
      { Ctx::G q{cn, c.H(ag + "kv_w"), static_cast<int>(Rc), 2 * hid, hid}; q.bias = c.F(ag + "kv_b"); q.out = kv; c.gemm(q); }
      float* q = ar.f(static_cast<size_t>(R4) * hid);
      c.small_linear(xn, R4, hid, c.F(ag + "q_w"), hid, c.F(ag + "q_b"), UDB_ACT_NONE, nullptr, nullptr, q);
      float* at = ar.f(static_cast<size_t>(R4) * hid);
      float* scratch = ar.f(static_cast<size_t>(B) * 16 * 4 * (hid + 2));
      if (!c.dry && !c.rc)
        c.done(udb_cross_attn_small(q, c.F("cam.pos"), kv, at, scratch, B, 4, 4 * nq + 4, hid, 1.0f / sqrtf(static_cast<float>(hid)), st));
      float* t2 = ar.f(static_cast<size_t>(R4) * hid);
      c.small_linear(at, R4, hid, c.F(ag + "out_w"), hid, c.F(ag + "out_b"), UDB_ACT_NONE, c.F(ag + "ls1"), cl, t2);
      t = cam_mlp(c, ag + "mlp", t2, R4, hid, cf.expansion * hid, hid, t2, c.F(ag + "ls2"));
    }
    for (int i = 0; i < 2; ++i) {
      const std::string ly = idx("cam.l%d.", i);
      float* xn = ar.f(static_cast<size_t>(R4) * hid);
      float* cn = ar.f(static_cast<size_t>(R4) * hid);
      c.layernorm(t, 1, xn, 1, c.F(ly + "nxw"), c.F(ly + "nxb"), R4, hid, 1e-5f);
      c.layernorm(t, 1, cn, 1, c.F(ly + "ncw"), c.F(ly + "ncb"), R4, hid, 1e-5f);
      float* q = ar.f(static_cast<size_t>(R4) * hid);
      float* kv = ar.f(static_cast<size_t>(R4) * 2 * hid);
      c.small_linear(xn, R4, hid, c.F(ly + "q_w"), hid, c.F(ly + "q_b"), UDB_ACT_NONE, nullptr, nullptr, q);
      c.small_linear(cn, R4, hid, c.F(ly + "kv_w"), 2 * hid, c.F(ly + "kv_b"), UDB_ACT_NONE, nullptr, nullptr, kv);
      float* a4 = ar.f(static_cast<size_t>(R4) * hid);
      if (!c.dry && !c.rc) c.done(udb_camera_attn4_f32(q, kv, c.F("cam.pos"), a4, B, hid, cf.heads, st));
      float* t2 = ar.f(static_cast<size_t>(R4) * hid);
      c.small_linear(a4, R4, hid, c.F(ly + "out_w"), hid, c.F(ly + "out_b"), UDB_ACT_NONE, c.F(ly + "ls1"), t, t2);
      t = cam_mlp(c, ly + "mlp", t2, R4, hid, cf.expansion * hid, hid, t2, c.F(ly + "ls2"));
    }
    float* xo = cam_mlp(c, "cam.out", t, R4, hid, 2 * hid, 1, nullptr, nullptr);       // [B*4, 1] == [B, 4]
    // the result must survive the release below: copy into a slot allocated before the mark is not possible with a bump
    // arena, so keep the camera scratch alive instead (0.3 GB at B=16) -- x4 points into it
    x4 = xo;
    (void)m;
  }
  if (!c.dry && !c.rc)
    c.done(udb_v1_camera_intrinsics(x4, a.intrinsics, B, net_h, net_w, static_cast<float>(g.ratio), g.pad_l, g.pad_t, a.skip_camera, intr4,
                                    a.out_intrinsics, k4_points, st));

  c.tap("intr4", intr4, sizeof(float) * B * 4);
  // ---- ray embeddings at the three decoder levels (decoder.py:203-220)
  stage.next("udb_v1:ray_embeddings");
  float* emb[3];
  {
    float shk[81];
    for (int l = 0; l <= 8; ++l)
      for (int mo = 0; mo <= 8; ++mo) {
        double k = 0.0;
        if (mo <= l) {
          double ratio_f = 1.0;                       // (l-m)! / (l+m)!
          for (int t = l - mo + 1; t <= l + mo; ++t) ratio_f /= t;
          k = sqrt((2 * l + 1) / (4.0 * M_PI) * ratio_f) * (mo > 0 ? sqrt(2.0) : 1.0);
        }
        shk[l * 9 + mo] = static_cast<float>(k);
      }
    const char* names[3] = {"rays.16.", "rays.8.", "rays.4."};
    for (int s = 0; s < 3; ++s) {
      const int gh = hc << s, gw = wc << s, Cs = hid >> s;
      const long long R = static_cast<long long>(B) * gh * gw;
      emb[s] = ar.f(R * Cs);
      const size_t m = ar.mark();
      __half* r = ar.h(R * 128);
      __half* m1 = ar.h(R * 384);
      if (!c.dry && !c.rc) {
        udb_v1_rays_t p;
        memset(&p, 0, sizeof(p));
        p.intr4 = intr4; p.B = B; p.net_h = net_h; p.net_w = net_w; p.gh = gh; p.gw = gw;
        p.ln_w = c.F(std::string(names[s]) + "ln_w"); p.ln_b = c.F(std::string(names[s]) + "ln_b"); p.out = r;
        memcpy(p.sh_k, shk, sizeof(shk));
        c.done(udb_v1_rays_sh81(&p, st));
      }
      const std::string n = names[s];
      c.expect2(n + "w1", 384, 128);
      { Ctx::G q{r, c.H(n + "w1"), static_cast<int>(R), 384, 128}; q.bias = c.F(n + "b1"); q.act = UDB_ACT_GELU; q.out = m1; c.gemm(q); }
      { Ctx::G q{m1, c.H(n + "w2"), static_cast<int>(R), Cs, 384}; q.bias = c.F(n + "b2"); q.out = emb[s]; q.out_f32 = 1; c.gemm(q); }
      ar.release(m);
    }
  }

  // ---- depth head (decoder.py:222-300)
  stage.next("udb_v1:depth_head_16");
  float* lat16 = ar.f(Rq * hid);
  {
    const size_t m = ar.mark();
    __half* f16l = ar.h(Rq * hid);
    { Ctx::G q{featcat, c.H("fcc_w"), static_cast<int>(Rq), hid, 4 * hid}; q.bias = c.F("fcc_b"); q.out = f16l; c.gemm(q); }
    __half* hN = ar.h(Rq * hid);
    __half* md = ar.h(Rq * 2 * hid);
    c.ln16(f16l, 0, hN, "lat.nw", "lat.nb", Rq, hid, 1e-5f);
    { Ctx::G q{hN, c.H("lat.w1"), static_cast<int>(Rq), 2 * hid, hid}; q.bias = c.F("lat.b1"); q.act = UDB_ACT_GELU; q.out = md; c.gemm(q); }
    { Ctx::G q{md, c.H("lat.w2"), static_cast<int>(Rq), hid, 2 * hid}; q.bias = c.F("lat.b2"); q.out = lat16; q.out_f32 = 1; c.gemm(q); }
    ar.release(m);
  }
  c.tap("emb16", emb[0], sizeof(float) * Rq * hid);
  c.tap("lat16_init", lat16, sizeof(float) * Rq * hid);
  dense_attn_block(c, "agg16.", lat16, B, nq, hid, tokens, 0, 4 * nq, tokens_pos);
  c.tap("lat16_agg", lat16, sizeof(float) * Rq * hid);
  dense_attn_block(c, "prompt.", lat16, B, nq, hid, emb[0], 1, nq, nullptr);
  c.tap("lat16_prompt", lat16, sizeof(float) * Rq * hid);
  for (int i = 0; i < cf.dec_depths[0]; ++i) mh_attn_block(c, idx("l16.%d.", i), lat16, B, nq, hid, cf.heads, emb[0], false);
  c.tap("lat16", lat16, sizeof(float) * Rq * hid);

  float* outs[3];
  float* lat = lat16;
  const char* ups[3] = {"up8.", "up4.", "up2."};
  const char* lys[3] = {"", "l8.%d.", "l4.%d."};
  const char* ons[3] = {"out8", "out4", "out2"};
  int ch = hc, cw = wc, C = hid;
  for (int s = 0; s < 3; ++s) {
    stage.next(s == 0 ? "udb_v1:up8" : (s == 1 ? "udb_v1:layers_8+up4" : "udb_v1:layers_4+up2"));
    if (s > 0)
      for (int i = 0; i < cf.dec_depths[s]; ++i) mh_attn_block(c, idx(lys[s], i), lat, B, ch * cw, C, cf.heads >> s, emb[s], true);
    const long long Rn = static_cast<long long>(B) * 4 * ch * cw;
    float* nxt = ar.f(Rn * (C / 2));
    __half* nxt16 = ar.h(Rn * (C / 2));
    outs[s] = ar.f(Rn);
    conv_upsample(c, ups[s], lat, emb[s], B, ch, cw, C, nxt, nxt16);
    if (!c.dry && !c.rc)
      c.done(udb_conv3x3_c1_exp(nxt16, c.F(std::string(ons[s]) + ".w"), static_cast<float>(c.S(std::string(ons[s]) + ".b")), outs[s], B, 2 * ch, 2 * cw,
                                C / 2, st));
    c.tap(s == 0 ? "lat8" : (s == 1 ? "lat4" : "lat2"), nxt, sizeof(float) * Rn * (C / 2));
    c.tap(ons[s], outs[s], sizeof(float) * Rn);
    lat = nxt;
    ch *= 2; cw *= 2; C /= 2;
  }

  // ---- post-processing (unidepthv1.py:66-94,352-366)
  stage.next("udb_v1:postprocess");
  float* mean = ar.f(static_cast<size_t>(B) * net_h * net_w);
  if (!c.dry && !c.rc) c.done(udb_v1_mean_maps(outs[0], outs[1], outs[2], mean, B, hc, wc, net_h, net_w, st));
  if (!c.dry && !c.rc) {
    udb_v1_postprocess_t p;
    memset(&p, 0, sizeof(p));
    p.mean = mean; p.k4 = k4_points; p.B = B; p.net_h = net_h; p.net_w = net_w;
    p.pad_l = g.pad_l; p.pad_r = g.pad_r; p.pad_t = g.pad_t; p.pad_b = g.pad_b; p.H = a.H; p.W = a.W;
    p.out_depth = a.out_depth; p.out_points = a.out_points;
    c.done(udb_v1_postprocess(&p, st));
  }
  if (!c.rc && ar.overflow) { set_error("engine_v1: workspace too small (%zu bytes needed)", ar.peak); return 1; }
  return c.rc;
}

}  // namespace udb

using namespace udb;

extern "C" {

int udb_v1_create(const udb_v1_config_t* cfg, udb_engine_v1** out) {
  if (!cfg || !out) { set_error("udb_v1_create: null argument"); return 1; }
  for (int i = 0; i < 4; ++i)
    if (cfg->dims[i] <= 0 || cfg->dims[i] % 64 || cfg->dims[i] > 1536 || cfg->depths[i] <= 0) {
      set_error("udb_v1_create: stage %d (depth %d, width %d): widths must be multiples of 64 up to 1536", i, cfg->depths[i], cfg->dims[i]);
      return 1;
    }
  if (cfg->hidden != 512 || cfg->heads != 8) {
    set_error("udb_v1_create: decoder hidden %d / heads %d not supported (512 / 8: 64-wide heads at every level)", cfg->hidden, cfg->heads);
    return 1;
  }
  if (cfg->net_h < 64 || cfg->net_w < 64) { set_error("udb_v1_create: network shape %dx%d too small", cfg->net_h, cfg->net_w); return 1; }
  udb_engine_v1* e = new udb_engine_v1();
  e->cfg = *cfg;
  *out = e;
  return 0;
}

int udb_v1_create_vit(const udb_v1_config_t* cfg, int32_t enc_heads, udb_engine_v1** out) {
  if (!cfg || !out) { set_error("udb_v1_create_vit: null argument"); return 1; }
  const int D = cfg->dims[0];
  for (int i = 0; i < 4; ++i)
    if (cfg->dims[i] != D || cfg->depths[i] <= 0) {
      set_error("udb_v1_create_vit: range %d (depth %d, width %d): the four widths must equal the embedding width and every "
                "range needs a block", i, cfg->depths[i], cfg->dims[i]);
      return 1;
    }
  if (D <= 0 || D % 64 || D > 1536 || enc_heads <= 0 || D / enc_heads != 64 || D % enc_heads) {
    set_error("udb_v1_create_vit: encoder width %d / heads %d: needs 64-wide heads and a width up to 1536", D, enc_heads);
    return 1;
  }
  if (cfg->net_h % 14 || cfg->net_w % 14) { set_error("udb_v1_create_vit: network shape %dx%d is not a multiple of 14", cfg->net_h, cfg->net_w); return 1; }
  if (udb_v1_create(cfg, out)) return 1;
  (*out)->vit_heads = enc_heads;
  return 0;
}

void udb_v1_destroy(udb_engine_v1* e) { delete e; }

int udb_v1_geometry(int32_t H, int32_t W, int32_t net_h, int32_t net_w, udb_v1_geometry_t* out) {
  if (!out || H <= 0 || W <= 0 || net_h <= 0 || net_w <= 0) { set_error("udb_v1_geometry: bad argument"); return 1; }
  const V1Geom g = v1_geometry(H, W, net_h, net_w);      // the function run_v1 uses
  out->resized_h = g.rh; out->resized_w = g.rw;
  out->pad_l = g.pad_l; out->pad_r = g.pad_r; out->pad_t = g.pad_t; out->pad_b = g.pad_b;
  out->ratio = g.ratio;
  return 0;
}

int udb_v1_set_weight(udb_engine_v1* e, const char* name, const void* dev_ptr, const int64_t* shape, int32_t ndim, int32_t dtype) {
  if (!e || !name || !dev_ptr || ndim < 0 || ndim > 4) { set_error("udb_v1_set_weight: bad argument"); return 1; }
  if (reinterpret_cast<uintptr_t>(dev_ptr) & 15) { set_error("udb_v1_set_weight(%s): pointer must be 16-byte aligned", name); return 1; }
  Weight w;
  w.p = dev_ptr; w.dtype = dtype; w.ndim = ndim;
  for (int i = 0; i < ndim; ++i) w.shape[i] = shape[i];
  e->w[name] = w;
  return 0;
}

int udb_v1_set_scalar(udb_engine_v1* e, const char* name, double value) {
  if (!e || !name) { set_error("udb_v1_set_scalar: bad argument"); return 1; }
  e->scalars[name] = value;
  return 0;
}

size_t udb_v1_workspace_bytes(udb_engine_v1* e, int32_t B, int32_t H, int32_t W) {
  if (!e || B <= 0 || H <= 0 || W <= 0) { set_error("udb_v1_workspace_bytes: bad argument"); return 0; }
  udb_infer_v1_args_t a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.W = W;
  Arena ar(nullptr, 0);
  if (run_v1(e, a, ar, nullptr)) return 0;
  char key[96];
  snprintf(key, sizeof(key), "%d,%d,%d", B, H, W);
  e->ws_need[key] = ar.peak + 256;
  return ar.peak + 256;
}

int udb_infer_v1(udb_engine_v1* e, const udb_infer_v1_args_t* a, void* stream) {
  if (!e || !a || !a->rgb || !a->workspace) { set_error("udb_infer_v1: null argument"); return 1; }
  if (!a->out_intrinsics || !a->out_points || !a->out_depth) { set_error("udb_infer_v1: all three output pointers are required"); return 1; }
  if (a->skip_camera && !a->intrinsics) { set_error("udb_infer_v1: skip_camera needs intrinsics"); return 1; }
  char key[96];
  snprintf(key, sizeof(key), "%d,%d,%d", a->B, a->H, a->W);
  auto need = e->ws_need.find(key);
  if (need == e->ws_need.end()) { set_error("udb_infer_v1: shape %dx%dx%d not prepared; call udb_v1_workspace_bytes first", a->B, a->H, a->W); return 1; }
  if (a->workspace_bytes < need->second) {
    set_error("udb_infer_v1: workspace too small (%zu bytes given, %zu needed)", a->workspace_bytes, need->second);
    return 1;
  }
  if (reinterpret_cast<uintptr_t>(a->workspace) & 255) { set_error("udb_infer_v1: workspace must be 256-byte aligned"); return 1; }
  Arena ar(a->workspace, a->workspace_bytes);
  return run_v1(e, *a, ar, stream);
}

}  // extern "C"
