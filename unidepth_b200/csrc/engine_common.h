// Shared by the whole-path engines (engine.cu: UniDepthV2, engine_v1.cu: UniDepthV1): registered weights, the bump
// allocator over the caller's workspace, NVTX stage ranges and thin wrappers that fill the operator argument structs.
#pragma once
#include <cuda_fp16.h>
#include <math.h>
#include <string.h>

#include <string>
#include <unordered_map>
#include <vector>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: stage ranges for nsys / ncu --nvtx (no-ops when no tool is attached)

#include "common.h"

namespace udb {

// NVTX range per stage of the schedule (host-side: it brackets the enqueue of that stage's kernels)
struct Stage {
  bool open = false;
  void next(const char* name) {
    if (open) nvtxRangePop();
    nvtxRangePushA(name);
    open = true;
  }
  ~Stage() { if (open) nvtxRangePop(); }
};

struct Weight {
  const void* p = nullptr;
  int dtype = 0;
  int ndim = 0;
  int64_t shape[4] = {0, 0, 0, 0};
};

// registered operands / scalars: the part of an engine the schedule helpers (Ctx) need
struct EngineBase {
  std::unordered_map<std::string, Weight> w;
  std::unordered_map<std::string, double> scalars;
};

// ------------------------------------------------------------------------------------------ arena
struct Arena {
  uintptr_t base;
  size_t cap, off = 0, peak = 0;
  bool dry;
  bool overflow = false;
  Arena(void* p, size_t c) : base(reinterpret_cast<uintptr_t>(p)), cap(c), dry(p == nullptr) {}
  void* alloc(size_t bytes) {
    off = (off + 255) & ~size_t(255);
    const size_t at = off;
    off += bytes;
    if (off > peak) peak = off;
    if (!dry && off > cap) overflow = true;
    return reinterpret_cast<void*>(base + at);
  }
  size_t mark() const { return off; }
  void release(size_t m) { off = m; }
  __half* h(size_t n) { return static_cast<__half*>(alloc(n * 2)); }
  float* f(size_t n) { return static_cast<float*>(alloc(n * 4)); }
};

// ------------------------------------------------------------------------------------------ run context
struct Ctx {
  EngineBase* e;
  Arena* ar;
  void* st;
  bool dry;
  int rc = 0;

  const Weight* W(const std::string& name) {
    auto it = e->w.find(name);
    if (it == e->w.end()) {
      if (!rc) set_error("engine: packed tensor '%s' was not registered (udb_set_weight)", name.c_str());
      rc = 1;
      static const Weight none;
      return &none;
    }
    return &it->second;
  }
  const __half* H(const std::string& n) { return static_cast<const __half*>(W(n)->p); }
  const float* F(const std::string& n) { return static_cast<const float*>(W(n)->p); }
  double S(const std::string& n) {
    auto it = e->scalars.find(n);
    if (it == e->scalars.end()) {
      if (!rc) set_error("engine: scalar '%s' was not registered (udb_set_scalar)", n.c_str());
      rc = 1;
      return 0.0;
    }
    return it->second;
  }
  void done(int r) { if (r && !rc) rc = r; }
  // registered 2-D operand must have exactly this shape (a mis-packed weight would otherwise be read with the
  // wrong leading dimension and silently produce garbage)
  void expect2(const std::string& name, int64_t rows, int64_t cols) {
    const Weight* w = W(name);
    if (rc) return;
    if (w->ndim != 2 || w->shape[0] != rows || w->shape[1] != cols) {
      set_error("engine: packed tensor '%s' has shape [%lld, %lld] (ndim %d), expected [%lld, %lld]", name.c_str(),
                (long long)w->shape[0], (long long)w->shape[1], w->ndim, (long long)rows, (long long)cols);
      rc = 1;
    }
  }

  // out[row(m), :] = resid + gamma * act(a @ w^T + bias)     (ops.gemm)
  struct G {
    const void* a; const void* w; int M, N, K; int lda = 0, ldw = 0;
    const float* bias = nullptr; const float* gamma = nullptr; const void* resid = nullptr; int resid_f32 = 0;
    long long ldr = 0; void* out = nullptr; int out_f32 = 0; long long ldc = 0; void* out2 = nullptr; int out2_leaky = 1;
    int act = UDB_ACT_NONE; int rows_per_group = 0, group_stride = 0, row_offset = 0, resid_mod = 0, resid_row_offset = 0;
    int a_split_k = 0, out_split = 0;    // split-f16 precise mode (udb_gemm_t)
    float* ln_stats_out = nullptr; const float* ln_stats_in = nullptr; const float* ln_c1 = nullptr;   // fused LayerNorm (udb_gemm_t.ln_*)
    int ln_parts = 0, ln_part_cols = 0; float ln_eps = 0.f;
  };
  void gemm(const G& q) {
    if (dry || rc) return;
    udb_gemm_t g;
    memset(&g, 0, sizeof(g));
    g.a = q.a; g.w = q.w; g.M = q.M; g.N = q.N; g.K = q.K;
    g.lda = q.lda ? q.lda : q.K; g.ldw = q.ldw ? q.ldw : q.K;
    g.a_mode = UDB_A_MATRIX;
    g.bias = q.bias; g.gamma = q.gamma;
    g.resid = q.resid; g.resid_f32 = q.resid_f32; g.ldr = q.resid ? (q.ldr ? q.ldr : q.N) : 0;
    g.out = q.out; g.out_f32 = q.out_f32; g.ldc = q.ldc ? q.ldc : q.N;
    g.out2 = q.out2; g.out2_leaky = q.out2_leaky;
    g.act = q.act; g.store_mode = UDB_STORE_ROWS;
    g.rows_per_group = q.rows_per_group; g.group_stride = q.group_stride; g.row_offset = q.row_offset;
    g.resid_mod = q.resid_mod; g.resid_row_offset = q.resid_row_offset;
    g.a_split_k = q.a_split_k; g.out_split = q.out_split;
    g.ln_stats_out = q.ln_stats_out; g.ln_stats_in = q.ln_stats_in; g.ln_c1 = q.ln_c1;
    g.ln_parts = q.ln_parts; g.ln_part_cols = q.ln_part_cols; g.ln_eps = q.ln_eps;
    done(udb_gemm_f16(&g, st));
  }
  // ConvTranspose2d with kernel == stride == k as a GEMM with a pixel-shuffle store (ops.conv_transpose_ks)
  void conv_transpose(const void* x, int M, int K, const void* w, int k, int cout, int h, int ww, const float* bias,
                      const void* resid, int resid_f32, void* out, int out_f32, void* out2, int out2_leaky, int pad) {
    if (dry || rc) return;
    udb_gemm_t g;
    memset(&g, 0, sizeof(g));
    g.a = x; g.w = w; g.M = M; g.N = k * k * cout; g.K = K; g.lda = K; g.ldw = K;
    g.a_mode = UDB_A_MATRIX;
    g.bias = bias; g.resid = resid; g.resid_f32 = resid_f32;
    g.out = out; g.out_f32 = out_f32; g.ldc = cout; g.out2 = out2; g.out2_leaky = out2_leaky;
    g.store_mode = UDB_STORE_CONVT;
    g.ct_k = k; g.ct_cout = cout; g.ct_h = h; g.ct_w = ww; g.ct_pad = pad;
    done(udb_gemm_f16(&g, st));
  }
  // 3x3 zero-padded convolution over NHWC f16 (ops.conv3x3, tile 8x16)
  void conv3x3(const void* x, int B, int H, int Wd, int C, const void* w, int N, const float* bias, int act,
               const float* gamma, const void* resid, int resid_f32, void* out, int out_f32, void* out2, int out2_leaky) {
    if (dry || rc) return;
    udb_gemm_t g;
    memset(&g, 0, sizeof(g));
    g.a = x; g.w = w; g.M = B * H * Wd; g.N = N; g.K = 9 * C; g.lda = C; g.ldw = 9 * C;
    g.a_mode = UDB_A_CONV3X3;
    g.conv_B = B; g.conv_H = H; g.conv_W = Wd; g.conv_C = C; g.conv_inH = H; g.conv_inW = Wd; g.conv_off = -1;
    g.conv_TH = 8; g.conv_TW = 16; g.conv_cstride = C; g.conv_coff = 0;
    g.bias = bias; g.gamma = gamma; g.act = act; g.store_mode = UDB_STORE_CONVTILE;
    g.out = out; g.out_f32 = out_f32; g.ldc = N;
    g.resid = resid; g.resid_f32 = resid_f32; g.ldr = resid ? N : 0;
    g.out2 = out2; g.out2_leaky = out2_leaky;
    done(udb_gemm_f16(&g, st));
  }
  void conv_halo(const void* x, int B, int H, int Wd, int C, int cstride, int coff, const void* w, int cout,
                 const float* bias, int act, void* out, const float* head_w, float head_b, float head_add, float* head_out) {
    if (dry || rc) return;
    udb_conv_halo_t c;
    memset(&c, 0, sizeof(c));
    c.x = x; c.w = w; c.bias = bias; c.B = B; c.H = H; c.W = Wd; c.C = C; c.cstride = cstride; c.coff = coff;
    c.cout = cout; c.act = act; c.out = out; c.ldc = cout;
    c.head_w = head_w; c.head_b = head_b; c.head_add = head_add; c.head_out = head_out;
    done(udb_conv3x3_halo_f16(&c, st));
  }
  void attention(const void* q, const void* k, const void* v, void* out, int B, int heads, int sq, int sk, int ldq,
                 int ldk, int ldv, int ldo, int q0, int k0, int v0, float scale, int lo_in = 0, int lo_out = 0) {
    if (dry || rc) return;
    udb_attn_t a;
    memset(&a, 0, sizeof(a));
    a.q = q; a.k = k; a.v = v; a.out = out; a.B = B; a.heads = heads; a.seq_q = sq; a.seq_k = sk; a.head_dim = 64;
    a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo; a.q_col0 = q0; a.k_col0 = k0; a.v_col0 = v0; a.o_col0 = 0;
    a.scale = scale;
    if (lo_in) { a.split = 1; a.lo_off_q = a.lo_off_k = a.lo_off_v = lo_in; a.lo_off_o = lo_out; }
    done(udb_attention_f16(&a, st));
  }
  void layernorm(const void* in, int in_f32, void* out, int out_f32, const float* w, const float* b, int rows, int dim,
                 float eps, int rows_per_group = 0, int group_stride = 0, int row_offset = 0, int dim_valid = 0,
                 int out_split = 0) {
    if (dry || rc) return;
    udb_layernorm_t p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.in_f32 = in_f32; p.out = out; p.out_f32 = out_f32; p.weight = w; p.bias = b;
    p.rows = rows; p.dim = dim; p.ld_in = dim; p.ld_out = out_split ? 2 * dim : dim;
    p.rows_per_group = rows_per_group; p.group_stride = group_stride; p.row_offset = row_offset; p.eps = eps;
    p.dim_valid = dim_valid;
    p.out_split = out_split;
    done(udb_layernorm(&p, st));
  }
  void small_linear(const float* x, int M, int K, const float* w, int N, const float* bias, int act, const float* gamma,
                    const float* resid, float* y, int ldx = 0, int ldy = 0, int ldr = 0) {
    if (dry || rc) return;
    udb_small_linear_t p;
    memset(&p, 0, sizeof(p));
    p.x = x; p.w = w; p.bias = bias; p.gamma = gamma; p.resid = resid; p.y = y; p.M = M; p.N = N; p.K = K; p.act = act;
    p.ldx = ldx ? ldx : K; p.ldy = ldy ? ldy : N; p.ldr = resid ? (ldr ? ldr : N) : 0;
    done(udb_small_linear_f32(&p, st));
  }
};

// LN -> Linear -> GELU -> Linear (+ gamma, + residual), fp32, camera head (layers/mlp.py:9-35)
static inline float* cam_mlp(Ctx& c, const std::string& pre, const float* x, int rows, int hid, int mid, int out_dim,
                      const float* resid, const float* gamma) {
  float* y = c.ar->f(static_cast<size_t>(rows) * hid);
  c.layernorm(x, 1, y, 1, c.F(pre + ".nw"), c.F(pre + ".nb"), rows, hid, 1e-5f);
  float* z = c.ar->f(static_cast<size_t>(rows) * mid);
  c.small_linear(y, rows, hid, c.F(pre + ".w1"), mid, c.F(pre + ".b1"), UDB_ACT_GELU, nullptr, nullptr, z);
  float* o = c.ar->f(static_cast<size_t>(rows) * out_dim);
  c.small_linear(z, rows, mid, c.F(pre + ".w2"), out_dim, c.F(pre + ".b2"), UDB_ACT_NONE, gamma, resid, o);
  return o;
}

// Scratch of vit_block, owned by the caller: h [B*T, D] (unused with fuse), qkv [B*T, 3D], att [B*T, D], mid [B*T, 4D]
// (each x2 in split mode); x16 / stats: the f16 copy of the residual stream and its per-part LayerNorm statistics (fuse only).
struct VitScratch {
  __half* h;
  __half* qkv;
  __half* att;
  __half* mid;
  __half* x16;
  float* stats;
  int ln_parts, ln_pc;
};

// One DINOv2 block on the f32 residual stream x [B*T, D] (metadinov2/block.py:84-109): LN -> qkv -> attention (64-wide
// heads) -> proj (ls1, +x) -> LN -> fc1 (GELU) -> fc2 (ls2, +x), with the operands blocks.<i>.* under prefix `b`.
// sp: split-f16 precise mode (every operand a hi/lo pair, weights [N, 3K]); fuse: LayerNorm folded into qkv / fc1, whose
// inputs are the x16 copy + statistics written by the GEMMs that update x.  Shared by the V2 engine and V1's ViT encoder.
static inline void vit_block(Ctx& c, const std::string& b, float* x, int B, int T, int D, int heads, bool sp, bool fuse,
                             const VitScratch& s) {
  const size_t BT = static_cast<size_t>(B) * T;
  const int sx = sp ? 2 : 1;
  const int kx = sp ? 3 : 1;          // logical K multiplier of a split operand
  const int ln_parts = s.ln_parts, ln_pc = s.ln_pc;
  __half *h = s.h, *qkv = s.qkv, *att = s.att, *mid = s.mid, *x16 = s.x16;
  float* stats = s.stats;
  // a weight packed for another mode (or transposed) must be refused, not read with the wrong leading dimension
  c.expect2(b + (fuse ? "qkv_wf" : "qkv_w"), 3 * D, D * kx);
  c.expect2(b + (fuse ? "fc1_wf" : "fc1_w"), 4 * D, D * kx);
  c.expect2(b + "proj_w", D, D * kx);
  c.expect2(b + "fc2_w", D, 4 * D * kx);
  if (fuse) {
    Ctx::G q{x16, c.H(b + "qkv_wf"), static_cast<int>(BT), 3 * D, D};
    q.bias = c.F(b + "qkv_c2"); q.ln_stats_in = stats; q.ln_c1 = c.F(b + "qkv_c1"); q.ln_parts = ln_parts; q.ln_part_cols = ln_pc;
    q.ln_eps = 1e-6f; q.out = qkv; c.gemm(q);
  } else {
    c.layernorm(x, 1, h, 0, c.F(b + "n1w"), c.F(b + "n1b"), static_cast<int>(BT), D, 1e-6f, 0, 0, 0, 0, sp ? D : 0);
    Ctx::G q{h, c.H(b + "qkv_w"), static_cast<int>(BT), 3 * D, D * kx}; q.lda = D * sx; q.a_split_k = sp ? D : 0;
    q.bias = c.F(b + "qkv_b"); q.out = qkv; q.ldc = 3 * D * sx; q.out_split = sp ? 3 * D : 0; c.gemm(q);
  }
  c.attention(qkv, qkv, qkv, att, B, heads, T, T, 3 * D * sx, 3 * D * sx, 3 * D * sx, D * sx, 0, D, 2 * D, 0.125f,
              sp ? 3 * D : 0, sp ? D : 0);
  { Ctx::G q{att, c.H(b + "proj_w"), static_cast<int>(BT), D, D * kx}; q.lda = D * sx; q.a_split_k = sp ? D : 0;
    q.bias = c.F(b + "proj_b"); q.gamma = c.F(b + "ls1");
    q.resid = x; q.resid_f32 = 1; q.out = x; q.out_f32 = 1;
    if (fuse) { q.out2 = x16; q.out2_leaky = 0; q.ln_stats_out = stats; q.ln_parts = ln_parts; q.ln_part_cols = ln_pc; }
    c.gemm(q); }
  if (fuse) {
    Ctx::G q{x16, c.H(b + "fc1_wf"), static_cast<int>(BT), 4 * D, D};
    q.bias = c.F(b + "fc1_c2"); q.ln_stats_in = stats; q.ln_c1 = c.F(b + "fc1_c1"); q.ln_parts = ln_parts; q.ln_part_cols = ln_pc;
    q.ln_eps = 1e-6f; q.act = UDB_ACT_GELU; q.out = mid; c.gemm(q);
  } else {
    c.layernorm(x, 1, h, 0, c.F(b + "n2w"), c.F(b + "n2b"), static_cast<int>(BT), D, 1e-6f, 0, 0, 0, 0, sp ? D : 0);
    Ctx::G q{h, c.H(b + "fc1_w"), static_cast<int>(BT), 4 * D, D * kx}; q.lda = D * sx; q.a_split_k = sp ? D : 0;
    q.bias = c.F(b + "fc1_b"); q.act = UDB_ACT_GELU;
    q.out = mid; q.ldc = 4 * D * sx; q.out_split = sp ? 4 * D : 0; c.gemm(q);
  }
  { Ctx::G q{mid, c.H(b + "fc2_w"), static_cast<int>(BT), D, 4 * D * kx}; q.lda = 4 * D * sx; q.a_split_k = sp ? 4 * D : 0;
    q.bias = c.F(b + "fc2_b"); q.gamma = c.F(b + "ls2");
    q.resid = x; q.resid_f32 = 1; q.out = x; q.out_f32 = 1;
    if (fuse) { q.out2 = x16; q.out2_leaky = 0; q.ln_stats_out = stats; q.ln_parts = ln_parts; q.ln_part_cols = ln_pc; }
    c.gemm(q); }
}

static inline std::string idx(const char* fmt, int i) {
  char b[64];
  snprintf(b, sizeof(b), fmt, i);
  return b;
}
static inline std::string idx2(const char* fmt, int i, int j) {
  char b[64];
  snprintf(b, sizeof(b), fmt, i, j);
  return b;
}

}  // namespace udb
