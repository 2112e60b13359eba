// Whole-path engine behind udb_create / udb_set_weight / udb_workspace_bytes / udb_infer_v2
// (include/udb.h): the host-side schedule of UniDepthV2.infer as one C call that only enqueues the
// kernels of this library on the caller's stream.  Reference call stack it replaces:
//   UniDepthV2.infer            unidepth/models/unidepthv2/unidepthv2.py:239-339
//     get_paddings / get_resize_factor                                  :36-77
//     encode_decode -> pixel_encoder (DINOv2)   backbones/metadinov2/*  dinov2.py:306-347, block.py:84-109
//                   -> pixel_decoder            unidepthv2/decoder.py:405-462 (camera head :85-111,
//                      rays :361-403, ray embedding :234-253, prompts :255-260, process :262-282,
//                      depth / confidence heads :284-313)
//     _postprocess                                                      :80-108
// Host code only (no kernels here); scratch memory comes from the caller's workspace through a bump
// allocator, so the same function run with a null workspace sizes it.
#include "engine_common.h"

namespace udb {

struct ShapeTables {       // per (gh, gw): engine-owned device tables
  float* pos = nullptr;    // [1 + gh*gw, D] cls row + bicubic-resized grid
  float* scales = nullptr; // [hidden/2]
};

constexpr int PATCH = 14;

}  // namespace udb

struct udb_engine : udb::EngineBase {
  udb_config_t cfg;
  std::unordered_map<long long, udb::ShapeTables> tables;
  std::unordered_map<std::string, size_t> ws_need;   // "B,H,W,level" -> bytes (filled by udb_workspace_bytes)
};

namespace udb {

// ------------------------------------------------------------------------------------------ geometry
// unidepthv2.py:36-58 (Python float == C double; int() truncates toward zero)
static inline int floordiv2(int v) { return v >= 0 ? v / 2 : -((-v + 1) / 2); }   // Python's v // 2

static void paddings(int H, int W, double lo, double hi, udb_geometry_t* g) {
  const double ratio = static_cast<double>(W) / H;
  const double target = fmin(hi, fmax(lo, ratio));
  g->pad_l = g->pad_r = g->pad_t = g->pad_b = 0;
  if (ratio > target) {
    const int h_new = static_cast<int>(W / target);
    g->pad_t = floordiv2(h_new - H);
    g->pad_b = h_new - H - g->pad_t;
    g->padded_h = h_new;
    g->padded_w = W;
  } else {
    const int w_new = static_cast<int>(H * target);
    g->pad_l = floordiv2(w_new - W);
    g->pad_r = w_new - W - g->pad_l;
    g->padded_h = H;
    g->padded_w = w_new;
  }
}

// unidepthv2.py:61-77 and the resolution_level bounds :247-262
static int resize(const udb_config_t& c, int level, udb_geometry_t* g) {
  double lo = c.pixels_min, hi = c.pixels_max;
  if (level >= 0) {
    if (level >= 10) { set_error("resolution_level should be in [0, 10)"); return 1; }
    const double interval = (hi - lo) / 10;
    const double l2 = level * interval + lo, h2 = (level + 1) * interval + lo;
    lo = l2;
    hi = h2;
  }
  const double n_ori = static_cast<double>(g->padded_w) * g->padded_h;
  const double target = fmin(hi, fmax(lo, n_ori));
  g->factor = pow(target / n_ori, 0.5);
  const int new_w = static_cast<int>(g->padded_w * g->factor);
  const int new_h = static_cast<int>(g->padded_h * g->factor);
  g->net_h = static_cast<int>(ceil(static_cast<double>(new_h) / PATCH)) * PATCH;
  g->net_w = static_cast<int>(ceil(static_cast<double>(new_w) / PATCH)) * PATCH;
  g->gh = g->net_h / PATCH;
  g->gw = g->net_w / PATCH;
  return 0;
}

// ------------------------------------------------------------------------------------------ the schedule
static int run(udb_engine* e, const udb_infer_args_t& a, const udb_geometry_t& g, const ShapeTables& tb, Arena& ar,
               void* st) {
  const udb_config_t& cf = e->cfg;
  Ctx c{e, &ar, st, ar.dry};
  const int B = a.B, nh = g.net_h, nw = g.net_w, gh = g.gh, gw = g.gw;
  const int N = gh * gw, T = N + 1, D = cf.embed_dim, hid = cf.hidden;
  const size_t BN = static_cast<size_t>(B) * N, BT = static_cast<size_t>(B) * T;

  // ---- a2/a3/a4: pre-process + patch embedding + cls / position rows
  Stage stage;
  stage.next("udb:preprocess+patch_embed");
  // Split-f16 precise mode (udb_set_scalar("precision", 1)): every f16 GEMM operand of the ENCODER is a hi/lo pair and
  // the weights are packed [N, 3K] = [hi | hi | lo] (udb_gemm_t.a_split_k); attention runs in the fp32 kernel.  The
  // cls tokens / camera head are fp32 anyway, so the intrinsics then carry no f16 operand rounding at all.
  const bool sp = e->scalars.count("precision") && e->scalars["precision"] == 1.0;
  const int sx = sp ? 2 : 1;
  // Fused LayerNorm (udb_set_scalar("fuse_ln", 1), default f16 mode): norm1 / norm2 never run as their own pass.  The GEMM
  // that updates the residual stream (patch embed, attn.proj, mlp.fc2) also writes the f16 copy of its rows and their
  // per-part statistics; qkv / fc1 read that copy with LayerNorm-folded weights (udb_gemm_t.ln_*; block.py:84-109).
  const bool fuse = !sp && e->scalars.count("fuse_ln") && e->scalars["fuse_ln"] == 1.0;
  const int ln_bn = D % 256 == 0 ? 256 : (D % 192 == 0 ? 192 : (D % 128 == 0 ? 128 : 64));   // udb_gemm_f16's tile width for N = D
  const int ln_parts = D / ln_bn * 2, ln_pc = ln_bn / 2;
  __half* x16 = fuse ? ar.h(BT * D) : nullptr;
  float* stats = fuse ? ar.f(BT * ln_parts * 2) : nullptr;
  __half* patches = ar.h(BN * 640 * sx);
  if (!c.dry) {
    udb_preprocess_t p;
    memset(&p, 0, sizeof(p));
    p.rgb = a.rgb; p.rgb_is_u8 = a.rgb_is_u8; p.normalize = a.normalize; p.B = B; p.H = a.H; p.W = a.W;
    p.pad_l = g.pad_l; p.pad_r = g.pad_r; p.pad_t = g.pad_t; p.pad_b = g.pad_b; p.net_h = nh; p.net_w = nw;
    p.patches = patches; p.ldp = 640 * sx; p.split = sp ? 1 : 0;
    c.done(udb_preprocess_patchify(&p, st));
  }
  float* x = ar.f(BT * D);           // fp32 residual stream
  {
    Ctx::G q{patches, c.H("patch_w"), static_cast<int>(BN), D, sp ? 3 * 640 : 640};
    q.lda = 640 * sx; q.a_split_k = sp ? 640 : 0;
    q.bias = c.F("patch_b"); q.resid = tb.pos; q.resid_f32 = 1; q.ldr = D; q.out = x; q.out_f32 = 1;
    q.rows_per_group = N; q.group_stride = T; q.row_offset = 1; q.resid_mod = N; q.resid_row_offset = 1;
    c.expect2("patch_w", D, sp ? 3 * 640 : 640);
    if (fuse) { q.out2 = x16; q.out2_leaky = 0; q.ln_stats_out = stats; q.ln_parts = ln_parts; q.ln_part_cols = ln_pc; }
    c.gemm(q);
    if (!c.dry && !c.rc)
      c.done(fuse ? udb_set_cls_rows_ln(x, x16, stats, c.F("cls"), tb.pos, B, T, D, ln_parts, ln_pc, st)
                  : udb_set_cls_rows(x, c.F("cls"), tb.pos, B, T, D, st));
  }

  // ---- a5-a8: transformer blocks, taps through the final norm
  stage.next("udb:encoder_blocks");
  __half* feats[4];
  float* clss[4];
  for (int l = 0; l < 4; ++l) { feats[l] = ar.h(BN * D); clss[l] = ar.f(static_cast<size_t>(B) * D); }
  {
    const size_t m = ar.mark();
    __half* h = fuse ? nullptr : ar.h(BT * D * sx);
    __half* qkv = ar.h(BT * 3 * D * sx);
    __half* att = ar.h(BT * D * sx);
    __half* mid = ar.h(BT * 4 * D * sx);
    const VitScratch vs{h, qkv, att, mid, x16, stats, ln_parts, ln_pc};
    int tap = 0;
    for (int i = 0; i < cf.depth; ++i) {
      vit_block(c, idx("blocks.%d.", i), x, B, T, D, cf.enc_heads, sp, fuse, vs);
      if (tap < 4 && i + 1 == cf.taps[tap]) {
        c.layernorm(x, 1, feats[tap], 0, c.F("norm_w"), c.F("norm_b"), static_cast<int>(BN), D, 1e-5f, N, T, 1);
        c.layernorm(x, 1, clss[tap], 1, c.F("norm_w"), c.F("norm_b"), B, D, 1e-5f, 1, T, 0);
        ++tap;
      }
    }
    if (tap != 4 && !c.rc) { set_error("engine: taps must be 4 increasing block indices <= depth"); c.rc = 1; }
    ar.release(m);
  }

  stage.next("udb:adapters+camera_head");
  // ---- a9: adapters (features f32 = the prompt blocks' residual; cls tokens -> camera tokens)
  float* Fl[4];
  for (int l = 0; l < 4; ++l) {
    Fl[l] = ar.f(BN * hid);
    Ctx::G q{feats[l], c.H(idx("adapt.%d.w", l)), static_cast<int>(BN), hid, D};
    q.bias = c.F(idx("adapt.%d.b", l)); q.out = Fl[l]; q.out_f32 = 1;
    c.gemm(q);
  }
  float* tokens = ar.f(static_cast<size_t>(B) * 4 * hid);
  for (int l = 0; l < 4; ++l)
    c.small_linear(clss[l], B, D, c.F(idx("cam_adapt.%d.w", l)), hid, c.F(idx("cam_adapt.%d.b", l)), UDB_ACT_NONE, nullptr,
                   nullptr, tokens + l * hid, D, 4 * hid, 0);

  // ---- a10: camera head, fp32 (decoder.py:85-111)
  const int R4 = B * 4;
  float* t = cam_mlp(c, "cam.project", tokens, R4, hid, hid, hid, nullptr, nullptr);
  for (int k = 1; k <= 2; ++k) {
    const std::string ag = idx("cam.agg%d", k);
    float* xn = ar.f(static_cast<size_t>(R4) * hid);
    float* cn = ar.f(static_cast<size_t>(R4) * hid);
    c.layernorm(t, 1, xn, 1, c.F(ag + ".nxw"), c.F(ag + ".nxb"), R4, hid, 1e-5f);
    c.layernorm(t, 1, cn, 1, c.F(ag + ".ncw"), c.F(ag + ".ncb"), R4, hid, 1e-5f);
    float* q = ar.f(static_cast<size_t>(R4) * hid);
    float* kv = ar.f(static_cast<size_t>(R4) * 2 * hid);
    c.small_linear(xn, R4, hid, c.F(ag + ".q"), hid, nullptr, UDB_ACT_NONE, nullptr, nullptr, q);
    c.small_linear(cn, R4, hid, c.F(ag + ".kv"), 2 * hid, nullptr, UDB_ACT_NONE, nullptr, nullptr, kv);
    float* a4 = ar.f(static_cast<size_t>(R4) * hid);
    if (!c.dry && !c.rc) c.done(udb_camera_attn4_f32(q, kv, c.F("cam.pos"), a4, B, hid, cf.dec_heads, st));
    float* t2 = ar.f(static_cast<size_t>(R4) * hid);
    c.small_linear(a4, R4, hid, c.F(ag + ".out"), hid, nullptr, UDB_ACT_NONE, c.F(ag + ".ls1"), t, t2);
    t = cam_mlp(c, ag + ".mlp", t2, R4, hid, cf.expansion * hid, hid, t2, c.F(ag + ".ls2"));
  }
  float* x4 = cam_mlp(c, "cam.pinhole", t, R4, hid, hid, 1, nullptr, nullptr);   // [B*4,1] == [B,4]
  float* intr4 = ar.f(static_cast<size_t>(B) * 4);
  float* k_net = ar.f(static_cast<size_t>(B) * 9);
  if (!c.dry && !c.rc)
    c.done(udb_camera_intrinsics(x4, B, nh, nw, static_cast<float>(g.factor), g.pad_l, g.pad_t, intr4, k_net, a.intrinsics, st));

  stage.next("udb:ray_embedding+prompt_blocks");
  // ---- a11/a12: rays (predicted K, or the caller's pinhole K) -> Fourier embedding on the patch grid
  const float* ray_intr = intr4;
  if (a.camera_k && !a.camera_rays) {
    float* gt4 = ar.f(static_cast<size_t>(B) * 4);
    if (!c.dry && !c.rc) c.done(udb_camera_adjust_k(a.camera_k, B, static_cast<float>(g.factor), g.pad_l, g.pad_t, gt4, st));
    ray_intr = gt4;
  }
  float* remb = ar.f(BN * hid);
  if (!c.dry && !c.rc) {
    udb_ray_embed_t p;
    memset(&p, 0, sizeof(p));
    p.intr4 = ray_intr; p.rays_in = a.camera_rays; p.scales = a.ray_scales ? a.ray_scales : tb.scales;
    p.B = B; p.net_h = nh; p.net_w = nw; p.gh = gh; p.gw = gw; p.bands = hid / 2; p.out = remb; p.out_f32 = 1;
    c.done(udb_ray_embed(&p, st));
  }

  // ---- a13: prompt blocks (cross attention to the ray embedding + MLP), fp16 residual out
  __half* cond[4];
  for (int l = 0; l < 4; ++l) cond[l] = ar.h(BN * hid);
  const int hd = hid / cf.dec_heads;          // true head dim; packed weights are zero-padded to 64
  const int hp = cf.dec_heads * 64;
  {
    const size_t m = ar.mark();
    __half* xn = ar.h(BN * hid);
    __half* cn = ar.h(BN * hid);
    __half* qb = ar.h(BN * hp);
    __half* kvb = ar.h(BN * 2 * hp);
    __half* ab = ar.h(BN * hp);
    __half* mb = ar.h(BN * cf.expansion * hid);
    const float scale = static_cast<float>(pow(static_cast<double>(hd), -0.5));
    for (int l = 0; l < 4; ++l) {
      const std::string p = idx("prompt.%d.", l);
      c.layernorm(Fl[l], 1, xn, 0, c.F(p + "nxw"), c.F(p + "nxb"), static_cast<int>(BN), hid, 1e-5f);
      c.layernorm(remb, 1, cn, 0, c.F(p + "ncw"), c.F(p + "ncb"), static_cast<int>(BN), hid, 1e-5f);
      { Ctx::G q{xn, c.H(p + "q"), static_cast<int>(BN), hp, hid}; q.out = qb; c.gemm(q); }
      { Ctx::G q{cn, c.H(p + "kv"), static_cast<int>(BN), 2 * hp, hid}; q.out = kvb; c.gemm(q); }
      c.attention(qb, kvb, kvb, ab, B, cf.dec_heads, N, N, hp, 2 * hp, 2 * hp, hp, 0, 0, hp, scale);
      { Ctx::G q{ab, c.H(p + "out"), static_cast<int>(BN), hid, hp}; q.resid = Fl[l]; q.resid_f32 = 1; q.out = Fl[l];
        q.out_f32 = 1; c.gemm(q); }
      c.layernorm(Fl[l], 1, xn, 0, c.F(p + "mnw"), c.F(p + "mnb"), static_cast<int>(BN), hid, 1e-5f);
      { Ctx::G q{xn, c.H(p + "w1"), static_cast<int>(BN), cf.expansion * hid, hid}; q.bias = c.F(p + "b1");
        q.act = UDB_ACT_GELU; q.out = mb; c.gemm(q); }
      { Ctx::G q{mb, c.H(p + "w2"), static_cast<int>(BN), hid, cf.expansion * hid}; q.bias = c.F(p + "b2");
        q.resid = Fl[l]; q.resid_f32 = 1; q.out = cond[l]; c.gemm(q); }
    }
    ar.release(m);
  }

  stage.next("udb:upsampling_stages");
  // ---- a14/a15: latents + up-sampling stages (NHWC, fp32 residual + fp16 activated copy)
  { Ctx::G q{cond[0], c.H("lat_w"), static_cast<int>(BN), hid, hid}; q.bias = c.F("lat_b"); q.out = a.depth_features;
    q.out_f32 = 1; c.gemm(q); }
  const void* prev = a.depth_features;   // fp32 for stage 0, fp16 (up-sampled) afterwards
  int prev_f32 = 1;
  int cur_h = gh, cur_w = gw, c_hr = 0;
  for (int i = 0; i < cf.n_stages; ++i) {
    const std::string s = idx("ups.%d.", i);
    const int k = i == 0 ? 1 : 2 * i;
    const Weight* ctw = c.W(s + "ct_w");
    const int cout = static_cast<int>(ctw->shape[0]) / (k * k);
    const int oh = cur_h, ow = cur_w;
    const size_t px = static_cast<size_t>(B) * oh * ow;
    __half* nxt = nullptr;
    const int up_c = static_cast<int>(c.W(s + "up_w")->shape[0]);
    nxt = ar.h(px * 4 * up_c);             // this stage's output survives the scratch below
    const size_t m = ar.mark();
    float* lat = ar.f(px * cout);
    __half* act = ar.h(px * cout);
    __half* tmp = ar.h(px * cout);
    c.conv_transpose(cond[i + 1], static_cast<int>(BN), hid, ctw->p, k, cout, gh, gw, c.F(s + "ct_b"), prev, prev_f32, lat, 1,
                     act, 1, 0);
    for (int j = 0; j < cf.dec_depths[i]; ++j) {
      const std::string r = idx2("ups.%d.rcu.%d.", i, j);
      c.expect2(r + "w1", cout, 9 * cout);     // 3x3 only (layers/upsample.py:137-180 with kernel_size=3)
      c.expect2(r + "w2", cout, 9 * cout);
      c.conv3x3(act, B, oh, ow, cout, c.H(r + "w1"), cout, c.F(r + "b1"), UDB_ACT_LEAKY, nullptr, nullptr, 0, tmp, 0,
                nullptr, 1);
      c.conv3x3(tmp, B, oh, ow, cout, c.H(r + "w2"), cout, c.F(r + "b2"), UDB_ACT_NONE, c.F(r + "gamma"), lat, 1, lat, 1,
                act, j + 1 < cf.dec_depths[i] ? 1 : 0);
    }
    __half* u = ar.h(px * up_c);
    { Ctx::G q{act, c.H(s + "up_w"), static_cast<int>(px), up_c, cout}; q.bias = c.F(s + "up_b"); q.out = u; c.gemm(q); }
    if (!c.dry && !c.rc) c.done(udb_upsample2x_nhwc_f16(u, nxt, B, oh, ow, up_c, st));
    ar.release(m);
    prev = nxt;
    prev_f32 = 0;
    cur_h = 2 * oh;
    cur_w = 2 * ow;
    c_hr = up_c;
  }
  const int hh = cur_h, hw = cur_w;
  const size_t hpx = static_cast<size_t>(B) * hh * hw;

  stage.next("udb:depth+confidence_heads");
  // ---- a16/a17: depth + confidence heads (shared normalisation, merged LN->Linear GEMM written
  //      straight into the reflect-padded buffer the 3x3 "lr" convs read)
  __half* xhat = ar.h(hpx * c_hr);
  // real width of the last map (decoder.py:470-524: max(2*hidden / 2^n_stages, out_dim)); ViT-B stores its 96
  // channels zero-padded to 128
  const int nxt_last = (2 * hid) >> cf.n_stages;
  const int c_valid = nxt_last > cf.out_dim ? nxt_last : cf.out_dim;
  c.layernorm(prev, 0, xhat, 0, c.F("ln_ones"), c.F("ln_zeros"), static_cast<int>(hpx), c_hr, 1e-5f, 0, 0, 0,
              c_valid != c_hr ? c_valid : 0);
  const int n_mlp = static_cast<int>(c.W("head_mlp_w")->shape[0]);   // 2 * out_dim: [depth | confidence]
  __half* mp = ar.h(static_cast<size_t>(B) * (hh + 2) * (hw + 2) * n_mlp);
  c.conv_transpose(xhat, static_cast<int>(hpx), c_hr, c.H("head_mlp_w"), 1, n_mlp, hh, hw, c.F("head_mlp_b"), nullptr, 0, mp,
                   0, nullptr, 1, 1);
  if (!c.dry && !c.rc) c.done(udb_reflect_border_fill_nhwc_f16(mp, B, hh, hw, n_mlp, st));
  float* planes[2];
  for (int i = 0; i < 2; ++i) {
    const std::string hn = idx("heads.%d.", i);
    const int lr_c = static_cast<int>(c.W(hn + "lr_w")->shape[0]);
    planes[i] = ar.f(static_cast<size_t>(B) * nh * nw);
    const size_t m = ar.mark();
    __half* lr = ar.h(hpx * lr_c);
    c.conv_halo(mp, B, hh, hw, n_mlp / 2, n_mlp, i * (n_mlp / 2), c.H(hn + "lr_w"), lr_c, c.F(hn + "lr_b"), UDB_ACT_NONE, lr,
                nullptr, 0.f, 0.f, nullptr);
    __half* up = ar.h(static_cast<size_t>(B) * (nh + 2) * (nw + 2) * lr_c);
    if (!c.dry && !c.rc) c.done(udb_resize_ac_pad_nhwc_f16(lr, up, B, hh, hw, lr_c, nh, nw, 1, st));
    c.conv_halo(up, B, nh, nw, lr_c, lr_c, 0, c.H(hn + "hr_w"), 32, c.F(hn + "hr_b"), UDB_ACT_LEAKY, nullptr,
                c.F(hn + "head_w"), static_cast<float>(c.S(hn + "head_b")), static_cast<float>(c.S(hn + "add")), planes[i]);
    ar.release(m);
  }

  stage.next("udb:postprocess");
  // ---- a18: output assembly at the original resolution
  if (!c.dry && !c.rc) {
    udb_postprocess_t p;
    memset(&p, 0, sizeof(p));
    p.radius = planes[0]; p.confidence = planes[1]; p.intr4 = ray_intr; p.rays_in = a.camera_rays;
    p.B = B; p.net_h = nh; p.net_w = nw; p.padded_h = g.padded_h; p.padded_w = g.padded_w; p.pad_l = g.pad_l; p.pad_t = g.pad_t;
    p.H = a.H; p.W = a.W;
    p.out_confidence = a.confidence; p.out_radius = a.radius; p.out_depth = a.depth; p.out_points = a.points; p.out_rays = a.rays;
    c.done(udb_postprocess(&p, st));
  }
  if (!c.rc && ar.overflow) { set_error("engine: workspace too small (%zu bytes needed)", ar.peak); return 1; }
  return c.rc;
}

// torch.linspace(0, log2(max(gh,gw)//2), bands) then 2**x, float32 (positional_embedding.py:231-233).
// torch fills linspace symmetrically: start + i*step for the first half, end - (n-1-i)*step for the rest.
static void ray_scale_table(int gh, int gw, int bands, std::vector<float>& out) {
  const int mx = (gh > gw ? gh : gw) / 2;
  const float end = static_cast<float>(log2(static_cast<double>(mx)));
  const float step = bands > 1 ? end / static_cast<float>(bands - 1) : 0.f;
  out.resize(bands);
  for (int i = 0; i < bands; ++i) {
    const float v = i < bands / 2 ? step * i : end - step * (bands - 1 - i);
    out[i] = powf(2.0f, v);
  }
}

static const ShapeTables* prepare(udb_engine* e, const udb_geometry_t& g) {
  const long long key = (static_cast<long long>(g.gh) << 32) | static_cast<unsigned>(g.gw);
  auto it = e->tables.find(key);
  if (it != e->tables.end()) return &it->second;
  auto pw = e->w.find("pos");
  if (pw == e->w.end()) { set_error("engine: 'pos' must be registered before udb_workspace_bytes"); return nullptr; }
  const int D = e->cfg.embed_dim, m = e->cfg.pos_grid, N = g.gh * g.gw;
  ShapeTables tb;
  auto fail = [&tb](const char* why) -> const ShapeTables* {      // nothing half-built stays allocated
    if (why) set_error("%s", why);
    cudaFree(tb.pos);
    cudaFree(tb.scales);
    return nullptr;
  };
  if (cudaMalloc(&tb.pos, static_cast<size_t>(N + 1) * D * 4) != cudaSuccess ||
      cudaMalloc(&tb.scales, static_cast<size_t>(e->cfg.hidden / 2) * 4) != cudaSuccess)
    return fail("engine: cudaMalloc of the per-shape tables failed");
  const float* pos = static_cast<const float*>(pw->second.p);
  cudaMemcpy(tb.pos, pos, static_cast<size_t>(D) * 4, cudaMemcpyDeviceToDevice);   // cls position
  if (g.gh == m && g.gw == m) {
    cudaMemcpy(tb.pos + D, pos + D, static_cast<size_t>(N) * D * 4, cudaMemcpyDeviceToDevice);
  } else if (udb_posembed_bicubic(pos + D, m, D, tb.pos + D, g.gh, g.gw, nullptr)) {
    return fail(nullptr);                                          // the operator has set the error text
  }
  std::vector<float> sc;
  ray_scale_table(g.gh, g.gw, e->cfg.hidden / 2, sc);
  cudaMemcpy(tb.scales, sc.data(), sc.size() * 4, cudaMemcpyHostToDevice);
  if (cudaDeviceSynchronize() != cudaSuccess) return fail("engine: preparing the per-shape tables failed");
  return &(e->tables[key] = tb);
}

}  // namespace udb

using namespace udb;

extern "C" {

int udb_create(const udb_config_t* cfg, udb_engine** out) {
  if (!cfg || !out) { set_error("udb_create: null argument"); return 1; }
  if (cfg->embed_dim <= 0 || cfg->embed_dim % 64 || cfg->embed_dim / cfg->enc_heads != 64) {
    set_error("udb_create: encoder needs 64-wide heads (embed_dim %d, heads %d)", cfg->embed_dim, cfg->enc_heads);
    return 1;
  }
  const int hd = cfg->dec_heads > 0 ? cfg->hidden / cfg->dec_heads : 0;
  if (hd <= 0 || hd > 64) { set_error("udb_create: decoder head dim %d not supported", hd); return 1; }
  if (cfg->n_stages < 1 || cfg->n_stages > 4) { set_error("udb_create: n_stages %d out of range", cfg->n_stages); return 1; }
  udb_engine* e = new udb_engine();
  e->cfg = *cfg;
  *out = e;
  return 0;
}

void udb_destroy(udb_engine* e) {
  if (!e) return;
  for (auto& kv : e->tables) {
    cudaFree(kv.second.pos);
    cudaFree(kv.second.scales);
  }
  delete e;
}

int udb_set_weight(udb_engine* e, const char* name, const void* dev_ptr, const int64_t* shape, int32_t ndim, int32_t dtype) {
  if (!e || !name || !dev_ptr || ndim < 0 || ndim > 4) { set_error("udb_set_weight: bad argument"); return 1; }
  if (reinterpret_cast<uintptr_t>(dev_ptr) & 15) { set_error("udb_set_weight(%s): pointer must be 16-byte aligned", name); return 1; }
  Weight w;
  w.p = dev_ptr;
  w.dtype = dtype;
  w.ndim = ndim;
  for (int i = 0; i < ndim; ++i) w.shape[i] = shape[i];
  e->w[name] = w;
  return 0;
}

int udb_set_scalar(udb_engine* e, const char* name, double value) {
  if (!e || !name) { set_error("udb_set_scalar: bad argument"); return 1; }
  e->scalars[name] = value;
  return 0;
}

int udb_geometry(const udb_engine* e, int32_t H, int32_t W, int32_t level, udb_geometry_t* out) {
  if (!e || !out || H <= 0 || W <= 0) { set_error("udb_geometry: bad argument"); return 1; }
  if (level == UDB_LEVEL_NETWORK_ONLY) {
    // the caller's tensor IS the network input (forward_test / ONNX-style entry, unidepthv2.py:134-160,
    // export.py:27-45): no padding, no resize, outputs at the same resolution
    if (H % PATCH || W % PATCH) { set_error("network-only input %dx%d must be a multiple of %d", H, W, PATCH); return 1; }
    memset(out, 0, sizeof(*out));
    out->padded_h = out->net_h = H;
    out->padded_w = out->net_w = W;
    out->gh = H / PATCH;
    out->gw = W / PATCH;
    out->factor = 1.0;
    return 0;
  }
  paddings(H, W, e->cfg.ratio_min, e->cfg.ratio_max, out);
  return resize(e->cfg, level, out);
}

size_t udb_schedule_bytes(udb_engine* e, int32_t B, int32_t H, int32_t W, int32_t level) {
  if (!e || B <= 0) { set_error("udb_schedule_bytes: bad argument"); return 0; }
  udb_geometry_t g;
  if (udb_geometry(e, H, W, level, &g)) return 0;
  udb_infer_args_t a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.W = W; a.resolution_level = level;
  a.camera_k = reinterpret_cast<const float*>(16);   // the larger (GT-camera) variant, as udb_workspace_bytes sizes it
  const ShapeTables none;                            // a dry run only hands the table pointers on
  Arena ar(nullptr, 0);
  if (run(e, a, g, none, ar, nullptr)) return 0;
  return ar.peak + 256;
}

size_t udb_workspace_bytes(udb_engine* e, int32_t B, int32_t H, int32_t W, int32_t level) {
  udb_geometry_t g;
  if (udb_geometry(e, H, W, level, &g)) return 0;
  const ShapeTables* tb = prepare(e, g);
  if (!tb) return 0;
  udb_infer_args_t a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.W = W; a.resolution_level = level;
  a.camera_k = reinterpret_cast<const float*>(16);   // sized for the larger (GT-camera) variant
  Arena ar(nullptr, 0);
  if (run(e, a, g, *tb, ar, nullptr)) return 0;
  char key[96];
  snprintf(key, sizeof(key), "%d,%d,%d,%d", B, H, W, level);
  e->ws_need[key] = ar.peak + 256;
  return ar.peak + 256;
}

int udb_infer_v2(udb_engine* e, const udb_infer_args_t* a, void* stream) {
  if (!e || !a || !a->rgb || !a->workspace) { set_error("udb_infer_v2: null argument"); return 1; }
  if (!a->confidence || !a->intrinsics || !a->radius || !a->depth || !a->points || !a->rays || !a->depth_features) {
    set_error("udb_infer_v2: all seven output pointers are required");
    return 1;
  }
  udb_geometry_t g;
  if (udb_geometry(e, a->H, a->W, a->resolution_level, &g)) return 1;
  const long long key = (static_cast<long long>(g.gh) << 32) | static_cast<unsigned>(g.gw);
  auto it = e->tables.find(key);
  char wkey[96];
  snprintf(wkey, sizeof(wkey), "%d,%d,%d,%d", a->B, a->H, a->W, a->resolution_level);
  auto need = e->ws_need.find(wkey);
  if (it == e->tables.end() || need == e->ws_need.end()) {
    set_error("udb_infer_v2: shape %dx%dx%d (level %d) not prepared; call udb_workspace_bytes first", a->B, a->H, a->W,
              a->resolution_level);
    return 1;
  }
  if (a->workspace_bytes < need->second) {   // checked BEFORE anything is launched
    set_error("udb_infer_v2: workspace too small (%zu bytes given, %zu needed)", a->workspace_bytes, need->second);
    return 1;
  }
  Arena ar(a->workspace, a->workspace_bytes);
  if (reinterpret_cast<uintptr_t>(a->workspace) & 255) { set_error("udb_infer_v2: workspace must be 256-byte aligned"); return 1; }
  return run(e, *a, g, it->second, ar, stream);
}

}  // extern "C"
