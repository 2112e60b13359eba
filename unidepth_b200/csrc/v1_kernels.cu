// Kernels that only the UniDepthV1 / ConvNeXt path needs (BASELINE config 4; include/udb.h "UniDepthV1 operators"):
// depthwise 7x7, channel LayerNorm for ConvNeXt widths (with space-to-depth output for the k2 s2 downsample and an
// additive table for "tokens + positional embedding"), antialiased bilinear resampling, the fused ray -> SH-81 ->
// LayerNorm embedding, the small dense-attention pieces (row softmax, 4-query cross attention, Nystrom landmarks /
// pseudo-inverse matmuls), single-output 3x3 convolutions and the V1 pre / post-processing.  All HBM- or
// latency-bound CUDA-core work; the GEMM-shaped parts of V1 run on the tcgen05 kernels of gemm.cu / attention.cu.
#include <math.h>

#include "common.h"
#include "ptx.cuh"

namespace udb {

#define ST(s) reinterpret_cast<cudaStream_t>(s)

static inline int grid_1d(long long total, int block = 256) {
  long long g = (total + block - 1) / block;
  const long long cap = (long long)num_sms() * 32;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------------------------------
// Antialiased bilinear weights of ONE axis, exactly ATen's _compute_indices_min_size_weights_aa (UpSampleKernel.cpp;
// F.interpolate(mode="bilinear", align_corners=False, antialias=True)): triangle filter of half-width
// max(scale, 1) around scale*(i+0.5), window clipped to the input, weights renormalised.
// Returns xmin / xsize and the inverse weight sum; weight(j) = tri((j + xmin - center + 0.5) * invscale) * norm.
// ------------------------------------------------------------------------------------------------------------------
struct AAxis {
  int xmin, xsize;
  float center, invscale, norm;
  __device__ __forceinline__ float w(int j) const {
    const float x = fabsf(((float)(j + xmin) - center + 0.5f) * invscale);
    return x < 1.f ? (1.f - x) * norm : 0.f;
  }
};
__device__ __forceinline__ AAxis aa_axis(int i, int in_size, float scale) {
  AAxis a;
  const float support = scale >= 1.f ? scale : 1.f;
  a.center = scale * ((float)i + 0.5f);
  a.invscale = scale >= 1.f ? 1.f / scale : 1.f;
  a.xmin = max((int)(a.center - support + 0.5f), 0);
  a.xsize = min((int)(a.center + support + 0.5f), in_size) - a.xmin;
  float tot = 0.f;
  a.norm = 1.f;
  for (int j = 0; j < a.xsize; ++j) tot += a.w(j);
  a.norm = tot != 0.f ? 1.f / tot : 1.f;
  return a;
}

// ------------------------------------------------------------------------------------------------------------------
// V1 pre-processing (unidepthv1.py:49-63,298-317): u8 / f32 NCHW -> /255 -> ImageNet normalise -> antialiased bilinear
// to (rh, rw) -> zero pad to the fixed network shape -> PxP stride-P patch rows [B*gh*gw, LD] f16 (column
// c*P*P + py*P + px, 3*P*P used, the rest zero).  P = 4, LD = 64: the ConvNeXt stem conv's im2col (convnext.py:371-383);
// P = 14, LD = 640: the DINOv2 patch embedding's (V2's patch-GEMM operand layout).
// ------------------------------------------------------------------------------------------------------------------
template <int P, int LD>
__global__ void __launch_bounds__(256) v1_preprocess_kernel(const udb_v1_preprocess_t p, int gh, int gw, float sh, float sw) {
  constexpr int NV = LD / 8;                              // 8-column vectors per patch row
  const long long total = (long long)p.B * gh * gw * NV;
  const float mean[3] = {0.485f, 0.456f, 0.406f};
  const float stdv[3] = {0.229f, 0.224f, 0.225f};
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int v8 = (int)(idx % NV);
    const long long row = idx / NV;
    const int gx = (int)(row % gw), gy = (int)((row / gw) % gh), b = (int)(row / ((long long)gw * gh));
    float val[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = v8 * 8 + j;
      float acc = 0.f;
      if (col < 3 * P * P) {
        const int c = col / (P * P), py = (col / P) % P, px = col % P;
        const int Y = gy * P + py - p.pad_t, X = gx * P + px - p.pad_l;     // position in the resized image
        if (Y >= 0 && Y < p.rh && X >= 0 && X < p.rw) {
          const AAxis ay = aa_axis(Y, p.H, sh), ax = aa_axis(X, p.W, sw);
          for (int jy = 0; jy < ay.xsize; ++jy) {
            float r = 0.f;
            const long long base = (((long long)b * 3 + c) * p.H + (ay.xmin + jy)) * p.W + ax.xmin;
            for (int jx = 0; jx < ax.xsize; ++jx) {
              float t = p.rgb_is_u8 ? (float)__ldg(reinterpret_cast<const uint8_t*>(p.rgb) + base + jx)
                                    : __ldg(reinterpret_cast<const float*>(p.rgb) + base + jx);
              if (p.scale255) t = t / 255.0f;
              if (p.normalize) t = (t - mean[c]) / stdv[c];
              r += ax.w(jx) * t;
            }
            acc += ay.w(jy) * r;
          }
        }
      }
      val[j] = acc;
    }
    *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(p.patches) + row * LD + v8 * 8) =
        make_uint4(pack_half2(val[0], val[1]), pack_half2(val[2], val[3]), pack_half2(val[4], val[5]), pack_half2(val[6], val[7]));
  }
}

// ------------------------------------------------------------------------------------------------------------------
// LayerNorm over the channels for any width that is a multiple of 64 up to 1536 (ConvNeXt: 192 / 384 / 768 / 1536;
// timm LayerNorm2d == channels-last LayerNorm, convnext.py:252-263; eps 1e-6 in the encoder, 1e-5 in the decoder).
// One warp per row, lane owns element pairs.  Extras: an additive f32 table (in = x[row] + add[row % add_mod]) for
// "tokens + positional embedding" (decoder.py:92-94), and a space-to-depth output mapping that writes pixel (y, x) of
// an [B,H,W,C] map into row (b, y/2, x/2), columns ((y&1)*2 + (x&1))*C + c of the k2 s2 downsample's im2col matrix
// (odd trailing row / column dropped, as the strided conv does).
// ------------------------------------------------------------------------------------------------------------------
template <bool IN_F32, bool OUT_F32, int R, int NV>
__global__ void __launch_bounds__(256) layernorm_any_kernel(const udb_layernorm_any_t p) {
  // one warp normalises R consecutive rows; all loads of the R rows are issued before the first reduction (narrow rows
  // alone -- 192 channels = 384 B -- do not keep enough bytes in flight); NV = max float2 per lane per row
  const long long row0 = ((long long)blockIdx.x * 8 + (threadIdx.x >> 5)) * R;
  const int lane = threadIdx.x & 31;
  if (row0 >= p.rows) return;
  const int nv = p.dim >> 6;   // float2 per lane
  float2 x[R][NV];
  float s[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const long long row = row0 + r < p.rows ? row0 + r : p.rows - 1;
    s[r] = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      if (i < nv) {
        const int e = (lane + 32 * i) * 2;
        if (IN_F32) {
          x[r][i] = *reinterpret_cast<const float2*>(reinterpret_cast<const float*>(p.in) + row * p.ld_in + e);
        } else {
          x[r][i] = __half22float2(*reinterpret_cast<const __half2*>(reinterpret_cast<const __half*>(p.in) + row * p.ld_in + e));
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const long long row = row0 + r < p.rows ? row0 + r : p.rows - 1;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      if (i < nv) {
        if (p.add) {
          const float2 a = *reinterpret_cast<const float2*>(p.add + (row % p.add_mod) * p.dim + (lane + 32 * i) * 2);
          x[r][i].x += a.x;
          x[r][i].y += a.y;
        }
        s[r] += x[r][i].x + x[r][i].y;
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const long long row = row0 + r;
    const float mean = wsum(s[r]) / (float)p.dim;
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
      if (i < nv) v += (x[r][i].x - mean) * (x[r][i].x - mean) + (x[r][i].y - mean) * (x[r][i].y - mean);
    const float rstd = rsqrtf(wsum(v) / (float)p.dim + p.eps);
    if (row >= p.rows) continue;
    long long obase = row * p.ld_out;
    if (p.s2d_w > 0) {
      const int xw = (int)(row % p.s2d_w), yh = (int)((row / p.s2d_w) % p.s2d_h), b = (int)(row / ((long long)p.s2d_w * p.s2d_h));
      const int oh = p.s2d_h >> 1, ow = p.s2d_w >> 1;
      if ((yh >> 1) >= oh || (xw >> 1) >= ow) continue;
      obase = (((long long)b * oh + (yh >> 1)) * ow + (xw >> 1)) * p.ld_out + ((yh & 1) * 2 + (xw & 1)) * p.dim;
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      if (i < nv) {
        const int e = (lane + 32 * i) * 2;
        const float2 w = __ldg(reinterpret_cast<const float2*>(p.weight + e));
        const float2 bb = __ldg(reinterpret_cast<const float2*>(p.bias + e));
        const float y0 = (x[r][i].x - mean) * rstd * w.x + bb.x, y1 = (x[r][i].y - mean) * rstd * w.y + bb.y;
        if (OUT_F32) *reinterpret_cast<float2*>(reinterpret_cast<float*>(p.out) + obase + e) = make_float2(y0, y1);
        else *reinterpret_cast<uint32_t*>(reinterpret_cast<__half*>(p.out) + obase + e) = pack_half2(y0, y1);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Depthwise 7x7 convolution, zero padding 3, NHWC f16 -> NHWC f16 (+bias), f32 accumulation
// (convnext.py:208-211 `conv_dw`, layers/convnext.py:16-24 `dwconv`).  A block owns an 8x16-pixel tile of 64 channels:
// the 14x22 halo is staged once in shared memory (2.4x read amplification instead of 49x), each thread slides along 8
// consecutive x for one 4-channel group, so per dy it loads 14 inputs + 7 weights for 56 FMA4.
// ------------------------------------------------------------------------------------------------------------------
constexpr int DW_CB = 64;
constexpr int DW_PS = DW_CB + 4;   // pixel stride in halves (136 B): keeps the 8-byte row reads of a warp on distinct banks

// TW = tile width (16 or 8), tile height = 128 / TW: wide tiles have the smaller halo, narrow ones waste fewer pixels on the
// small late-stage maps (28x38, 14x19); the launcher picks the shape with the least padded area.
template <int TW>
__global__ void __launch_bounds__(256) dwconv7_kernel(const __half* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                                     __half* __restrict__ y, int H, int W, int C, int tiles_x) {
  constexpr int TH = 128 / TW, HH = TH + 6, HW = TW + 6;
  __shared__ __align__(16) __half tile[HH * HW * DW_PS];
  const int tx0 = (blockIdx.x % tiles_x) * TW, ty0 = (blockIdx.x / tiles_x) * TH;
  const int c0 = blockIdx.y * DW_CB, b = blockIdx.z;
  const __half* xb = x + (long long)b * H * W * C;
  for (int i = threadIdx.x; i < HH * HW * (DW_CB / 8); i += 256) {
    const int ch = i & 7, pix = i >> 3;
    const int hy = pix / HW, hx = pix - hy * HW;
    const int gy = ty0 + hy - 3, gx = tx0 + hx - 3;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (gy >= 0 && gy < H && gx >= 0 && gx < W) v = __ldg(reinterpret_cast<const uint4*>(xb + ((long long)gy * W + gx) * C + c0 + ch * 8));
    uint2* d = reinterpret_cast<uint2*>(tile + pix * DW_PS + ch * 8);      // 8-byte aligned (136 B pixel stride)
    d[0] = make_uint2(v.x, v.y);
    d[1] = make_uint2(v.z, v.w);
  }
  __syncthreads();
  const int cg = threadIdx.x & 15, pg = threadIdx.x >> 4;
  const int r = TW == 16 ? (pg >> 1) : pg, xh = TW == 16 ? (pg & 1) * 8 : 0;     // each thread: 8 consecutive x of one row
  uint64_t acc[8][2];          // packed f32x2: (c0,c1), (c2,c3)
  {
    const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + c0 + cg * 4));
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[i][0] = pack2(bv.x, bv.y); acc[i][1] = pack2(bv.z, bv.w); }
  }
#pragma unroll 1
  for (int dy = 0; dy < 7; ++dy) {
    uint64_t in[14][2];
#pragma unroll
    for (int i = 0; i < 14; ++i) {
      const uint2 u = *reinterpret_cast<const uint2*>(tile + ((r + dy) * HW + xh + i) * DW_PS + cg * 4);
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
      const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      in[i][0] = pack2(a.x, a.y);
      in[i][1] = pack2(c.x, c.y);
    }
#pragma unroll
    for (int dx = 0; dx < 7; ++dx) {
      const float4 wv = __ldg(reinterpret_cast<const float4*>(w + (long long)(dy * 7 + dx) * C + c0 + cg * 4));
      const uint64_t w0 = pack2(wv.x, wv.y), w1 = pack2(wv.z, wv.w);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        acc[i][0] = fma2(in[i + dx][0], w0, acc[i][0]);
        acc[i][1] = fma2(in[i + dx][1], w1, acc[i][1]);
      }
    }
  }
  const int gy = ty0 + r;
  if (gy < H) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int gx = tx0 + xh + i;
      if (gx < W) {
        float a0, a1, a2, a3;
        unpack2(acc[i][0], a0, a1);
        unpack2(acc[i][1], a2, a3);
        *reinterpret_cast<uint2*>(y + (((long long)b * H + gy) * W + gx) * C + c0 + cg * 4) = make_uint2(pack_half2(a0, a1), pack_half2(a2, a3));
      }
    }
  }
}

// running element-wise maximum over a stage's block outputs (decoder.py:371-374 `max_stack`): dst = first ? src : max(dst, src)
__global__ void __launch_bounds__(256) max_accum_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, long long n8, int first) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    uint4 s = src[i];
    if (!first) {
      const uint4 d = dst[i];
      __half2* sh = reinterpret_cast<__half2*>(&s);
      const __half2* dh = reinterpret_cast<const __half2*>(&d);
#pragma unroll
      for (int j = 0; j < 4; ++j) sh[j] = __hmax2(sh[j], dh[j]);
    }
    dst[i] = s;
  }
}

// ViT tap after one block (unidepthv1.py:322-326 + decoder.py:371-374): dst[b, n, :] = f16(x[b, 1+n, :] + x[b, 0, :]) on the
// first block of a range, max(dst, that) on the later ones; f16 rounding is monotone, so the running f16 max equals one
// rounding of the f32 max.  cls (optional): the f32 cls row x[b, 0, :] -> [B, D].  One thread per 8 channels (16-byte stores).
__global__ void __launch_bounds__(256) vit_tap_kernel(const float* __restrict__ x, uint4* __restrict__ dst, float* __restrict__ cls,
                                                      int N, int D, long long total, int first) {
  const int dv = D >> 3;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c8 = (int)(i % dv);
    const long long bn = i / dv;
    const long long b = bn / N, n = bn % N;
    const float* xc = x + b * (N + 1) * D + c8 * 8;
    const float4* pr = reinterpret_cast<const float4*>(xc + (n + 1) * D);
    const float4* pc = reinterpret_cast<const float4*>(xc);
    const float4 r0 = pr[0], r1 = pr[1], c0 = __ldg(pc), c1 = __ldg(pc + 1);
    uint4 v = make_uint4(pack_half2(r0.x + c0.x, r0.y + c0.y), pack_half2(r0.z + c0.z, r0.w + c0.w),
                         pack_half2(r1.x + c1.x, r1.y + c1.y), pack_half2(r1.z + c1.z, r1.w + c1.w));
    if (!first) {
      const uint4 d = dst[i];
      __half2* vh = reinterpret_cast<__half2*>(&v);
      const __half2* dh = reinterpret_cast<const __half2*>(&d);
#pragma unroll
      for (int j = 0; j < 4; ++j) vh[j] = __hmax2(vh[j], dh[j]);
    }
    dst[i] = v;
    if (cls && n == 0) {
      float4* o = reinterpret_cast<float4*>(cls + b * D + c8 * 8);
      o[0] = c0;
      o[1] = c1;
    }
  }
}

// spatial mean of an NHWC f32 map -> [B, C] f32 (ConvNeXt "cls tokens", convnext.py:471)
__global__ void __launch_bounds__(256) spatial_mean_kernel(const float* __restrict__ x, float* __restrict__ out, int HW, int C) {
  const int b = blockIdx.y;
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int part = threadIdx.x >> 5;   // 8 row groups
  __shared__ float red[8][33];
  float s = 0.f;
  if (c < C)
    for (int i = part; i < HW; i += 8) s += x[((long long)b * HW + i) * C + c];
  red[part][threadIdx.x & 31] = s;
  __syncthreads();
  if (part == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x & 31];
    out[(long long)b * C + c] = t / (float)HW;
  }
}

// antialiased bilinear resize of an NHWC f16 map (flat_interpolate, geometric.py:228-252): one thread per 8 channels
__global__ void __launch_bounds__(256) aa_resize_nhwc_kernel(const __half* __restrict__ in, __half* __restrict__ out, int B, int H, int W, int C,
                                                            int oh, int ow, float sh, float sw) {
  const int cv = C >> 3;
  const long long total = (long long)B * oh * ow * cv;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c8 = (int)(idx % cv);
    const long long pix = idx / cv;
    const int ox = (int)(pix % ow), oy = (int)((pix / ow) % oh), b = (int)(pix / ((long long)ow * oh));
    const AAxis ay = aa_axis(oy, H, sh), ax = aa_axis(ox, W, sw);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int jy = 0; jy < ay.xsize; ++jy) {
      float r[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = 0.f;
      for (int jx = 0; jx < ax.xsize; ++jx) {
        const uint4 u = *reinterpret_cast<const uint4*>(in + (((long long)b * H + ay.xmin + jy) * W + ax.xmin + jx) * C + c8 * 8);
        const __half2* h = reinterpret_cast<const __half2*>(&u);
        const float wx = ax.w(jx);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 f = __half22float2(h[q]);
          r[2 * q] += wx * f.x;
          r[2 * q + 1] += wx * f.y;
        }
      }
      const float wy = ay.w(jy);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += wy * r[j];
    }
    *reinterpret_cast<uint4*>(out + pix * C + c8 * 8) =
        make_uint4(pack_half2(acc[0], acc[1]), pack_half2(acc[2], acc[3]), pack_half2(acc[4], acc[5]), pack_half2(acc[6], acc[7]));
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Ray embedding of one decoder level (decoder.py:203-220): unit rays of the pinhole K at network resolution
// (generate_rays, geometric.py:13-45) are never materialised -- each token antialias-averages the analytic rays of its
// window (flat_interpolate), re-normalises, evaluates the 81 real spherical harmonics up to degree 8 by recurrence
// (rsh_cart_8, sht.py:833; same index l*(l+1)+m) and applies the MLP's input LayerNorm (81 wide, eps 1e-5).  Output
// f16 [B*gh*gw, 128], columns >= 81 zero (the projection GEMM's K is zero-extended).  One warp per token.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rays_sh81_kernel(const udb_v1_rays_t p) {
  const long long tok = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (tok >= (long long)p.B * p.gh * p.gw) return;
  const int gx = (int)(tok % p.gw), gy = (int)((tok / p.gw) % p.gh), b = (int)(tok / ((long long)p.gw * p.gh));
  const float fx = p.intr4[b * 4], fy = p.intr4[b * 4 + 1], cx = p.intr4[b * 4 + 2], cy = p.intr4[b * 4 + 3];
  const float sh = (float)p.net_h / (float)p.gh, sw = (float)p.net_w / (float)p.gw;
  const AAxis ay = aa_axis(gy, p.net_h, sh), ax = aa_axis(gx, p.net_w, sw);
  float rx = 0.f, ry = 0.f, rz = 0.f;
  const int taps = ay.xsize * ax.xsize;
  for (int t = lane; t < taps; t += 32) {
    const int jy = t / ax.xsize, jx = t % ax.xsize;
    const float dx = ((float)(ax.xmin + jx) + 0.5f - cx) / fx, dy = ((float)(ay.xmin + jy) + 0.5f - cy) / fy;
    const float inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + 1.0f), 1e-12f);
    const float wgt = ay.w(jy) * ax.w(jx);
    rx += wgt * dx * inv;
    ry += wgt * dy * inv;
    rz += wgt * inv;
  }
  rx = wsum(rx); ry = wsum(ry); rz = wsum(rz);
  {
    const float inv = 1.0f / fmaxf(sqrtf(rx * rx + ry * ry + rz * rz), 1e-12f);
    rx *= inv; ry *= inv; rz *= inv;
  }
  // every lane evaluates the recurrence (cheap, keeps the warp converged) and keeps the entries it stores
  float mine[3] = {0.f, 0.f, 0.f};
  float sum = 0.f, sq = 0.f;
  float A = 1.f, Bm = 0.f, pmm = 1.f;
  for (int m = 0; m <= 8; ++m) {
    if (m > 0) {
      const float a2 = rx * A - ry * Bm, b2 = rx * Bm + ry * A;
      A = a2; Bm = b2;
      pmm *= -(float)(2 * m - 1);
    }
    float pprev = 0.f, pcur = pmm;
    for (int l = m; l <= 8; ++l) {
      if (l == m + 1) { pprev = pcur; pcur = (float)(2 * m + 1) * rz * pcur; }
      else if (l > m + 1) { const float t = ((float)(2 * l - 1) * rz * pcur - (float)(l + m - 1) * pprev) / (float)(l - m); pprev = pcur; pcur = t; }
      const float k = p.sh_k[l * 9 + m];
      if (m == 0) {
        const float v = k * pcur;
        const int id = l * (l + 1);
        sum += v; sq += v * v;
        if ((id & 31) == lane) mine[id >> 5] = v;
      } else {
        const float va = k * A * pcur, vb = k * Bm * pcur;
        const int ia = l * (l + 1) + m, ib = l * (l + 1) - m;
        sum += va + vb; sq += va * va + vb * vb;
        if ((ia & 31) == lane) mine[ia >> 5] = va;
        if ((ib & 31) == lane) mine[ib >> 5] = vb;
      }
    }
  }
  const float mean = sum / 81.f;
  // two-pass variance from the stored entries (each lane holds up to 3 of the 81)
  float v = 0.f;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int id = lane + 32 * j;
    if (id < 81) v += (mine[j] - mean) * (mine[j] - mean);
  }
  (void)sq;
  const float rstd = rsqrtf(wsum(v) / 81.f + 1e-5f);
  __half* o = reinterpret_cast<__half*>(p.out) + tok * 128;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int id = lane + 32 * j;
    float y = 0.f;
    if (id < 81) y = (mine[j < 3 ? j : 0] - mean) * rstd * p.ln_w[id] + p.ln_b[id];
    o[id] = __float2half_rn(y);
  }
}

// V1 camera head tail (decoder.py:96-106,326-331; unidepthv1.py:88-91): x4 = (log fx', log fy', logit cx', logit cy') ->
// K at network resolution (intr4 = fx, fy, cx, cy) and the intrinsics returned to the caller (un-padded, / ratio).
// With GT intrinsics: K_net = K*ratio (+pads) (unidepthv1.py:56-62); skip_camera returns the GT K instead of the prediction.
__global__ void v1_camera_intrinsics_kernel(const float* x4, const float* gt_k, int B, int net_h, int net_w, float ratio, int pad_l, int pad_t,
                                            int skip_camera, float* intr4_rays, float* k_out, float* k4_points) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float fx = 0.f, fy = 0.f, cx = 0.f, cy = 0.f;
  if (x4) {
    const float half_max = (float)max(net_h, net_w) / 2.0f;
    fx = half_max * expf(x4[b * 4]);
    fy = half_max * expf(x4[b * 4 + 1]);
    cx = (1.0f / (1.0f + expf(-x4[b * 4 + 2]))) * (float)net_w;
    cy = (1.0f / (1.0f + expf(-x4[b * 4 + 3]))) * (float)net_h;
  }
  float rfx = fx, rfy = fy, rcx = cx, rcy = cy;     // K the rays are generated from
  if (gt_k) {
    rfx = gt_k[b * 9] * ratio;
    rfy = gt_k[b * 9 + 4] * ratio;
    rcx = gt_k[b * 9 + 2] * ratio + (float)pad_l;
    rcy = gt_k[b * 9 + 5] * ratio + (float)pad_t;
    if (skip_camera || !x4) { fx = rfx; fy = rfy; cx = rcx; cy = rcy; }
  }
  intr4_rays[b * 4] = rfx; intr4_rays[b * 4 + 1] = rfy; intr4_rays[b * 4 + 2] = rcx; intr4_rays[b * 4 + 3] = rcy;
  float* k = k_out + b * 9;
  k[0] = fx / ratio; k[1] = 0.f; k[2] = (cx - (float)pad_l) / ratio;
  k[3] = 0.f; k[4] = fy / ratio; k[5] = (cy - (float)pad_t) / ratio;
  k[6] = 0.f; k[7] = 0.f; k[8] = 1.f;
  // K the final back-projection uses on the ORIGINAL pixel grid (unidepthv1.py:354-356): the pre-processed GT K when one
  // was given (the reference does not undo its resize there), else the returned prediction
  float* kp = k4_points + b * 4;
  if (gt_k) { kp[0] = rfx; kp[1] = rfy; kp[2] = rcx; kp[3] = rcy; }
  else { kp[0] = k[0]; kp[1] = k[4]; kp[2] = k[2]; kp[3] = k[5]; }
}

// 4-query cross attention of the camera head (decoder.py:95, AttentionBlock num_heads=1): q f32 [B*nq, D] (+ q_pos), kv f16
// [B*nk, 2D] (k | v), out f32 [B*nq, D].  Keys are split over CA_SPLITS blocks per image (flash-decoding style): each block
// reads its slice of K and V ONCE for all queries and writes a partial (max, sum, weighted V); a second kernel merges.
constexpr int CA_SPLITS = 16, CA_MAXQ = 4;

__global__ void __launch_bounds__(256) cross_attn_partial_kernel(const float* __restrict__ q, const float* __restrict__ q_pos,
                                                                const __half* __restrict__ kv, float* __restrict__ part, int nq, int nk, int D,
                                                                float scale) {
  extern __shared__ float sm[];
  const int chunk = (nk + CA_SPLITS - 1) / CA_SPLITS;
  float* qs = sm;                       // [nq][D]
  float* sc = qs + nq * D;              // [nq][chunk]
  float* red = sc + nq * chunk;         // [nq][8] partial max / sum
  const int b = blockIdx.y, sp = blockIdx.x;
  const int j0 = sp * chunk, j1 = min(nk, j0 + chunk), n = max(j1 - j0, 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < nq * D; i += 256)
    qs[i] = (q[(long long)b * nq * D + i] + (q_pos ? q_pos[i] : 0.f)) * scale;
  __syncthreads();
  const __half* kb = kv + (long long)b * nk * 2 * D;
  for (int j = warp; j < n; j += 8) {
    float a[CA_MAXQ] = {0.f, 0.f, 0.f, 0.f};
    const __half* kr = kb + (long long)(j0 + j) * 2 * D;
    for (int d = lane * 8; d < D; d += 256) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(kr + d));
      const __half2* h = reinterpret_cast<const __half2*>(&u);
      float kf[8];
#pragma unroll
      for (int t = 0; t < 4; ++t) { const float2 f = __half22float2(h[t]); kf[2 * t] = f.x; kf[2 * t + 1] = f.y; }
#pragma unroll
      for (int qi = 0; qi < CA_MAXQ; ++qi)
        if (qi < nq) {
#pragma unroll
          for (int t = 0; t < 8; ++t) a[qi] = fmaf(qs[qi * D + d + t], kf[t], a[qi]);
        }
    }
#pragma unroll
    for (int qi = 0; qi < CA_MAXQ; ++qi)
      if (qi < nq) {
        const float v = wsum(a[qi]);
        if (lane == 0) sc[qi * chunk + j] = v;
      }
  }
  __syncthreads();
  // per query: max, exp, sum over this block's keys (warp qi handles query qi)
  if (warp < nq) {
    float m = -INFINITY;
    for (int j = lane; j < n; j += 32) m = fmaxf(m, sc[warp * chunk + j]);
    m = wmax(m);
    float l = 0.f;
    for (int j = lane; j < n; j += 32) {
      const float e = expf(sc[warp * chunk + j] - m);
      sc[warp * chunk + j] = e;
      l += e;
    }
    l = wsum(l);
    if (lane == 0) { red[warp * 2] = m; red[warp * 2 + 1] = l; }
  }
  __syncthreads();
  float* pb = part + ((long long)(b * CA_SPLITS + sp) * nq) * (D + 2);
  for (int d = threadIdx.x * 2; d < D; d += 512) {
    float acc[CA_MAXQ][2] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
    for (int j = 0; j < n; ++j) {
      const float2 vf = __half22float2(*reinterpret_cast<const __half2*>(kb + (long long)(j0 + j) * 2 * D + D + d));
#pragma unroll
      for (int qi = 0; qi < CA_MAXQ; ++qi)
        if (qi < nq) {
          const float pw = sc[qi * chunk + j];
          acc[qi][0] = fmaf(pw, vf.x, acc[qi][0]);
          acc[qi][1] = fmaf(pw, vf.y, acc[qi][1]);
        }
    }
    for (int qi = 0; qi < nq; ++qi) {
      pb[qi * (D + 2) + 2 + d] = acc[qi][0];
      pb[qi * (D + 2) + 2 + d + 1] = acc[qi][1];
    }
  }
  if (threadIdx.x < nq) {
    pb[threadIdx.x * (D + 2)] = n > 0 ? red[threadIdx.x * 2] : -INFINITY;
    pb[threadIdx.x * (D + 2) + 1] = n > 0 ? red[threadIdx.x * 2 + 1] : 0.f;
  }
}

__global__ void __launch_bounds__(256) cross_attn_merge_kernel(const float* __restrict__ part, float* __restrict__ out, int nq, int D) {
  const int b = blockIdx.y, qi = blockIdx.x;
  float m = -INFINITY;
  for (int s = 0; s < CA_SPLITS; ++s) m = fmaxf(m, part[((long long)(b * CA_SPLITS + s) * nq + qi) * (D + 2)]);
  float wgt[CA_SPLITS], tot = 0.f;
#pragma unroll
  for (int s = 0; s < CA_SPLITS; ++s) {
    const float* pp = part + ((long long)(b * CA_SPLITS + s) * nq + qi) * (D + 2);
    wgt[s] = expf(pp[0] - m);
    tot += wgt[s] * pp[1];
  }
  const float inv = 1.0f / tot;
  for (int d = threadIdx.x; d < D; d += 256) {
    float a = 0.f;
#pragma unroll
    for (int s = 0; s < CA_SPLITS; ++s) a = fmaf(wgt[s], part[((long long)(b * CA_SPLITS + s) * nq + qi) * (D + 2) + 2 + d], a);
    out[((long long)b * nq + qi) * D + d] = a * inv;
  }
}

// softmax over the first n_valid columns of f32 rows [rows, ld_in] -> f16 probabilities [rows, ld_out] (columns
// n_valid .. ld_out-1 zero): the P operand of the dense single-head attentions (aggregate_16 / prompt_camera).
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ s, __half* __restrict__ p, long long rows, int n_valid,
                                                          int ld_in, int ld_out, float scale) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* sr = s + row * ld_in;
  float m = -INFINITY;
  for (int j = lane; j < n_valid; j += 32) m = fmaxf(m, sr[j]);
  m = wmax(m);
  float tot = 0.f;
  for (int j = lane; j < n_valid; j += 32) tot += expf((sr[j] - m) * scale);
  tot = wsum(tot);
  const float inv = 1.0f / tot;
  __half* pr = p + row * ld_out;
  for (int j = lane; j < ld_out; j += 32) pr[j] = __float2half_rn(j < n_valid ? expf((sr[j] - m) * scale) * inv : 0.f);
}

// out[i] = a[i] + b[i] (f32, + optional f16 copy): `latents + rays_embedding` before each ConvUpsample (decoder.py:246-252)
__global__ void __launch_bounds__(256) add_f32_kernel(const float4* __restrict__ a, const float4* __restrict__ b, float4* __restrict__ o,
                                                     uint2* __restrict__ o16, long long n4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = a[i], y = b[i];
    const float4 r = make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
    if (o) o[i] = r;
    if (o16) o16[i] = make_uint2(pack_half2(r.x, r.y), pack_half2(r.z, r.w));
  }
}

// f32 rows -> f16 rows with independent row strides (cls tokens appended to the camera head's context, decoder.py:94)
__global__ void copy_rows_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, int groups, int rows_per_group, int D,
                                     long long dst_group_stride, long long dst_row0) {
  const long long total = (long long)groups * rows_per_group * D;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const long long r = i / D;
    const long long g = r / rows_per_group, rr = r % rows_per_group;
    dst[(g * dst_group_stride + dst_row0 + rr) * D + d] = __float2half_rn(src[i]);
  }
}

// 3x3 convolution with ONE output channel, zero padding, fused exp(clamp(., -10, 10)) (decoder.py:253,268,283,292-294
// `out8/out4/out2`): NHWC f16 in, f32 plane out.  One warp per output pixel, lanes over channel pairs.
template <int LPP>      // lanes per pixel = C / 8 (8, 16 or 32): each lane owns 8 channels (one 16-byte load per tap)
__global__ void __launch_bounds__(256) conv3x3_c1_kernel(const __half* __restrict__ x, const float* __restrict__ w, float bias, float* __restrict__ out,
                                                        int B, int H, int W, int C) {
  constexpr int PPW = 32 / LPP;                      // pixels per warp
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPP;
  const long long pix = ((long long)blockIdx.x * 8 + (threadIdx.x >> 5)) * PPW + lane / LPP;
  const bool live = pix < (long long)B * H * W;
  const long long pc = live ? pix : 0;
  const int px = (int)(pc % W), py = (int)((pc / W) % H), b = (int)(pc / ((long long)W * H));
  float a = 0.f;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int yy = py + t / 3 - 1, xx = px + t % 3 - 1;
    if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + (((long long)b * H + yy) * W + xx) * C + sub * 8));
    const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + t * C + sub * 8)), w1 = __ldg(reinterpret_cast<const float4*>(w + t * C + sub * 8 + 4));
    const __half2* h = reinterpret_cast<const __half2*>(&u);
    const float2 f0 = __half22float2(h[0]), f1 = __half22float2(h[1]), f2 = __half22float2(h[2]), f3 = __half22float2(h[3]);
    a = fmaf(f0.x, w0.x, fmaf(f0.y, w0.y, fmaf(f1.x, w0.z, fmaf(f1.y, w0.w, a))));
    a = fmaf(f2.x, w1.x, fmaf(f2.y, w1.y, fmaf(f3.x, w1.z, fmaf(f3.y, w1.w, a))));
  }
#pragma unroll
  for (int o = LPP / 2; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (live && sub == 0) out[pix] = expf(fminf(fmaxf(a + bias, -10.0f), 10.0f));
}

// ------------------------------------------------------------------------------------------------------------------
// Nystrom attention pieces (layers/nystrom_attention.py:22-84 -> xformers NystromAttention(num_landmarks=128); the
// restated algorithm is in oracle/unidepth_v1_oracle.py, PARITY UNPINNED).  Landmarks = segment means of q and k.
// q lives in qbuf [B*n, ldq] (cols h*64..), k in kvbuf [B*n, ldkv]; out f16 [B*128, 2*heads*64] = (q landmarks | k landmarks).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) nystrom_landmarks_kernel(const __half* __restrict__ q, int ldq, const __half* __restrict__ kv, int ldkv,
                                                              __half* __restrict__ out, int n, int heads, int m) {
  const int lm = blockIdx.x, h = blockIdx.y, b = blockIdx.z, d = threadIdx.x;
  const int seg = n / m, n_round = m - n % m;      // first n_round segments have `seg` rows, the rest seg + 1
  int start, len;
  if (n % m == 0 || lm < n_round) { start = lm * seg; len = seg; }
  else { start = n_round * seg + (lm - n_round) * (seg + 1); len = seg + 1; }
  float sq = 0.f, sk = 0.f;
  for (int r = 0; r < len; ++r) {
    const long long row = (long long)b * n + start + r;
    sq += __half2float(q[row * ldq + h * 64 + d]);
    sk += __half2float(kv[row * ldkv + h * 64 + d]);
  }
  __half* o = out + ((long long)b * m + lm) * (2 * heads * 64);
  o[h * 64 + d] = __float2half_rn(sq / (float)len);
  o[heads * 64 + h * 64 + d] = __float2half_rn(sk / (float)len);
}

// kernel_2 = softmax(q_landmarks . k_landmarks^T / sqrt(64)) per (b, head): f32 [B*heads, 128, 128].  One warp per row.
__global__ void __launch_bounds__(128) nystrom_k2_kernel(const __half* __restrict__ lmk, float* __restrict__ k2, int heads, int m) {
  const int bh = blockIdx.y, b = bh / heads, h = bh % heads;
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= m) return;
  const int ld = 2 * heads * 64;
  const __half* qr = lmk + ((long long)b * m + row) * ld + h * 64;
  float qv[2];
  qv[0] = __half2float(qr[lane * 2]);
  qv[1] = __half2float(qr[lane * 2 + 1]);
  float s[4];      // m == 128: 4 columns per lane
  float mx = -INFINITY;
  for (int j = 0; j < 4; ++j) {
    const int col = lane + 32 * j;
    const __half* kr = lmk + ((long long)b * m + col) * ld + heads * 64 + h * 64;
    float a = 0.f;
    for (int d = 0; d < 64; d += 2) {
      const float2 kf = __half22float2(*reinterpret_cast<const __half2*>(kr + d));
      const float q0 = __shfl_sync(0xffffffffu, qv[0], d >> 1), q1 = __shfl_sync(0xffffffffu, qv[1], d >> 1);
      a = fmaf(q0, kf.x, fmaf(q1, kf.y, a));
    }
    s[j] = a * 0.125f;
    mx = fmaxf(mx, s[j]);
  }
  mx = wmax(mx);
  float tot = 0.f;
  for (int j = 0; j < 4; ++j) { s[j] = expf(s[j] - mx); tot += s[j]; }
  tot = wsum(tot);
  for (int j = 0; j < 4; ++j) k2[((long long)bh * m + row) * m + lane + 32 * j] = s[j] / tot;
}

// Z0 = K^T / max_j(sum_i K[i][j]) (exact 1/||K||_1 initialisation of the Newton-Schulz iteration), per matrix
__global__ void __launch_bounds__(128) nystrom_pinv_init_kernel(const float* __restrict__ k2, float* __restrict__ z, int m) {
  const float* K = k2 + (long long)blockIdx.x * m * m;
  float* Z = z + (long long)blockIdx.x * m * m;
  __shared__ float red[4];
  const int j = threadIdx.x;      // m == 128 threads: column sums
  float cs = 0.f;
  for (int i = 0; i < m; ++i) cs += K[i * m + j];
  float mx = wmax(cs);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  const float inv = 1.0f / mx;
  for (int i = 0; i < m; ++i) Z[j * m + i] = K[i * m + j] * inv;     // Z[j][i] = K[i][j] / ||K||_1
}

// T = c*I - X over a batch of m x m matrices
__global__ void __launch_bounds__(256) eye_minus_kernel(const float* __restrict__ x, float* __restrict__ t, float c, int m, long long total) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i % ((long long)m * m));
    t[i] = ((e / m) == (e % m) ? c : 0.f) - x[i];
  }
}

// batched small matmul, f32:  C = diag * I + alpha * (A @ B), A [M,K], B [K,N] (f32, or f16 with row stride ldb),
// C [M,N] f32 or f16 with row stride ldc.
struct BmmArgs {
  const float* A; long long sA; int lda;
  const void* Bp; long long sB1, sB2; int ldb; int b_f16; int inner;   // batch index bh -> (bh / inner, bh % inner) for B and C strides
  void* C; long long sC1, sC2; int ldc; int c_f16;
  int M, N, K;
  float alpha, diag;
};
__global__ void __launch_bounds__(256) bmm_f32_kernel(const BmmArgs p) {
  // 64 x 64 output tile per block, 4 x 4 per thread, K in steps of 16 through shared memory
  __shared__ float As[16][64 + 4], Bs[16][64 + 4];
  const int bh = blockIdx.z, o = bh / p.inner, i2 = bh % p.inner;
  const float* A = p.A + (long long)bh * p.sA;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // outputs rows ty*4.., cols tx*4..
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < p.K; k0 += 16) {
    // A tile 64 x 16 (stored transposed [k][m]); B tile 16 x 64
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int idx = threadIdx.x + 256 * t;             // 1024 elements each
      const int am = idx >> 4, ak = idx & 15;
      const int mm = m0 + am, kk = k0 + ak;
      As[ak][am] = (mm < p.M && kk < p.K) ? A[(long long)mm * p.lda + kk] : 0.f;
      const int bk = idx >> 6, bn = idx & 63;
      const int kr = k0 + bk, nn = n0 + bn;
      float bv = 0.f;
      if (kr < p.K && nn < p.N) {
        const long long off = o * p.sB1 + i2 * p.sB2 + (long long)kr * p.ldb + nn;
        bv = p.b_f16 ? __half2float(reinterpret_cast<const __half*>(p.Bp)[off]) : reinterpret_cast<const float*>(p.Bp)[off];
      }
      Bs[bk][bn] = bv;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int mm = m0 + ty * 4 + i, nn = n0 + tx * 4 + j;
      if (mm < p.M && nn < p.N) {
        const float v = p.alpha * acc[i][j] + (mm == nn ? p.diag : 0.f);
        const long long off = o * p.sC1 + i2 * p.sC2 + (long long)mm * p.ldc + nn;
        if (p.c_f16) reinterpret_cast<__half*>(p.C)[off] = __float2half_rn(v);
        else reinterpret_cast<float*>(p.C)[off] = v;
      }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// V1 post-processing (unidepthv1.py:66-94,352-366).  Stage 1: the three exp'ed maps are antialias-resized to the
// network shape and averaged.  Stage 2: crop the paddings, antialias-resize to the original size -> depth (z), and
// back-project with (theta, phi) of the unit ray through each original pixel: x = z tan(theta) = z rx/rz,
// y = z / tan(phi) / cos(theta) (spherical_zbuffer_to_euclidean, geometric.py:57-73).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) v1_mean_maps_kernel(const float* __restrict__ o8, const float* __restrict__ o4, const float* __restrict__ o2,
                                                          float* __restrict__ mean, int B, int gh, int gw, int net_h, int net_w) {
  const long long total = (long long)B * net_h * net_w;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int X = (int)(idx % net_w), Y = (int)((idx / net_w) % net_h), b = (int)(idx / ((long long)net_w * net_h));
    float tot = 0.f;
#pragma unroll
    for (int lvl = 0; lvl < 3; ++lvl) {
      const int h = gh << (lvl + 1), w = gw << (lvl + 1);
      const float* src = (lvl == 0 ? o8 : (lvl == 1 ? o4 : o2)) + (long long)b * h * w;
      const AAxis ay = aa_axis(Y, h, (float)h / (float)net_h), ax = aa_axis(X, w, (float)w / (float)net_w);
      float acc = 0.f;
      for (int jy = 0; jy < ay.xsize; ++jy) {
        float r = 0.f;
        for (int jx = 0; jx < ax.xsize; ++jx) r += ax.w(jx) * src[(long long)(ay.xmin + jy) * w + ax.xmin + jx];
        acc += ay.w(jy) * r;
      }
      tot += acc;
    }
    mean[idx] = tot / 3.0f;
  }
}

__global__ void __launch_bounds__(256) v1_postprocess_kernel(const udb_v1_postprocess_t p) {
  const long long total = (long long)p.B * p.H * p.W;
  const int ch = p.net_h - p.pad_t - p.pad_b, cw = p.net_w - p.pad_l - p.pad_r;     // cropped size
  const float sh = (float)ch / (float)p.H, sw = (float)cw / (float)p.W;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int X = (int)(idx % p.W), Y = (int)((idx / p.W) % p.H), b = (int)(idx / ((long long)p.W * p.H));
    const AAxis ay = aa_axis(Y, ch, sh), ax = aa_axis(X, cw, sw);
    const float* src = p.mean + (long long)b * p.net_h * p.net_w;
    float z = 0.f;
    for (int jy = 0; jy < ay.xsize; ++jy) {
      float r = 0.f;
      for (int jx = 0; jx < ax.xsize; ++jx) r += ax.w(jx) * src[(long long)(p.pad_t + ay.xmin + jy) * p.net_w + p.pad_l + ax.xmin + jx];
      z += ay.w(jy) * r;
    }
    const float* k = p.k4 + b * 4;       // fx, fy, cx, cy of the K the points are generated with
    const float dx = ((float)X + 0.5f - k[2]) / k[0], dy = ((float)Y + 0.5f - k[3]) / k[1];
    const float inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + 1.0f), 1e-12f);
    const float rx = dx * inv, ry = dy * inv, rz = inv;
    const float theta = atan2f(rx, rz), phi = acosf(ry);
    const long long hw = (long long)p.H * p.W, pix = (long long)Y * p.W + X;
    p.out_depth[b * hw + pix] = z;
    p.out_points[(b * 3 + 0) * hw + pix] = z * tanf(theta);
    p.out_points[(b * 3 + 1) * hw + pix] = z / tanf(phi) / cosf(theta);
    p.out_points[(b * 3 + 2) * hw + pix] = z;
  }
}

}  // namespace udb

using namespace udb;

extern "C" {

int udb_v1_preprocess(const udb_v1_preprocess_t* p, void* stream) {
  if (p->net_h < 4 || p->net_w < 4) { set_error("udb_v1_preprocess: bad network shape"); return 1; }
  const int gh = (p->net_h - 4) / 4 + 1, gw = (p->net_w - 4) / 4 + 1;
  const float sh = (float)p->H / (float)p->rh, sw = (float)p->W / (float)p->rw;
  v1_preprocess_kernel<4, 64><<<grid_1d((long long)p->B * gh * gw * 8), 256, 0, ST(stream)>>>(*p, gh, gw, sh, sw);
  return check_launch("v1_preprocess_kernel");
}

int udb_v1_preprocess_vit(const udb_v1_preprocess_t* p, void* stream) {
  if (p->net_h < 14 || p->net_w < 14) { set_error("udb_v1_preprocess_vit: bad network shape"); return 1; }
  const int gh = p->net_h / 14, gw = p->net_w / 14;
  const float sh = (float)p->H / (float)p->rh, sw = (float)p->W / (float)p->rw;
  v1_preprocess_kernel<14, 640><<<grid_1d((long long)p->B * gh * gw * 80), 256, 0, ST(stream)>>>(*p, gh, gw, sh, sw);
  return check_launch("v1_preprocess_vit_kernel");
}

int udb_vit_tap_f16(const float* x, void* dst, float* cls, int32_t B, int32_t T, int32_t D, int32_t first, void* stream) {
  if (B <= 0 || T < 2 || D <= 0 || D % 8) { set_error("udb_vit_tap_f16: bad shape (B %d, T %d, D %d; D must be a multiple of 8)", B, T, D); return 1; }
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(cls)) & 15) {
    set_error("udb_vit_tap_f16: pointers must be 16-byte aligned");
    return 1;
  }
  const long long total = (long long)B * (T - 1) * (D / 8);
  vit_tap_kernel<<<grid_1d(total), 256, 0, ST(stream)>>>(x, reinterpret_cast<uint4*>(dst), cls, T - 1, D, total, first);
  return check_launch("vit_tap_kernel");
}

int udb_layernorm_any(const udb_layernorm_any_t* p, void* stream) {
  if (p->dim % 64 || p->dim > 1536 || p->dim <= 0) { set_error("udb_layernorm_any: dim %d unsupported (multiple of 64, <= 1536)", p->dim); return 1; }
  if (p->rows <= 0) return 0;
  note_work(0.0, (double)p->rows * p->dim * ((p->in_f32 ? 4 : 2) + (p->out_f32 ? 4 : 2)));
  // rows per warp by width: 4 up to 256 channels, 2 up to 768, 1 beyond (registers: R * dim / 32 floats)
#define UDB_LN_ANY(R_, NV_)                                                                                        \
  do {                                                                                                             \
    const int grid = (int)((p->rows + 8 * (R_) - 1) / (8 * (R_)));                                                 \
    if (p->in_f32 && p->out_f32) layernorm_any_kernel<true, true, R_, NV_><<<grid, 256, 0, ST(stream)>>>(*p);     \
    else if (p->in_f32) layernorm_any_kernel<true, false, R_, NV_><<<grid, 256, 0, ST(stream)>>>(*p);             \
    else if (p->out_f32) layernorm_any_kernel<false, true, R_, NV_><<<grid, 256, 0, ST(stream)>>>(*p);            \
    else layernorm_any_kernel<false, false, R_, NV_><<<grid, 256, 0, ST(stream)>>>(*p);                           \
  } while (0)
  if (p->dim <= 256) UDB_LN_ANY(4, 4);
  else if (p->dim <= 768) UDB_LN_ANY(2, 12);
  else UDB_LN_ANY(1, 24);
#undef UDB_LN_ANY
  return check_launch("layernorm_any_kernel");
}

int udb_dwconv7_nhwc_f16(const void* x, const float* w, const float* bias, void* y, int32_t B, int32_t H, int32_t W, int32_t C, void* stream) {
  if (C % DW_CB) { set_error("udb_dwconv7_nhwc_f16: C=%d must be a multiple of 64", C); return 1; }
  // 16x8 or 8x16 (W x H) pixel tiles: whichever pads the map less
  const long long area16 = (long long)((W + 15) / 16) * ((H + 7) / 8), area8 = (long long)((W + 7) / 8) * ((H + 15) / 16);
  note_work(2.0 * 49 * B * H * W * C, 4.0 * B * H * W * C);
  const __half* xh = reinterpret_cast<const __half*>(x);
  __half* yh = reinterpret_cast<__half*>(y);
  if (area16 <= area8) {
    const int tx = (W + 15) / 16, ty = (H + 7) / 8;
    dwconv7_kernel<16><<<dim3(tx * ty, C / DW_CB, B), 256, 0, ST(stream)>>>(xh, w, bias, yh, H, W, C, tx);
  } else {
    const int tx = (W + 7) / 8, ty = (H + 15) / 16;
    dwconv7_kernel<8><<<dim3(tx * ty, C / DW_CB, B), 256, 0, ST(stream)>>>(xh, w, bias, yh, H, W, C, tx);
  }
  return check_launch("dwconv7_kernel");
}

int udb_max_accum_f16(const void* src, void* dst, int64_t n, int32_t first, void* stream) {
  if (n % 8) { set_error("udb_max_accum_f16: n must be a multiple of 8"); return 1; }
  note_work(0.0, (first ? 4.0 : 6.0) * n);
  max_accum_kernel<<<grid_1d(n / 8), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), n / 8, first);
  return check_launch("max_accum_kernel");
}

int udb_spatial_mean_f32(const float* x, float* out, int32_t B, int32_t HW, int32_t C, void* stream) {
  dim3 grid((C + 31) / 32, B);
  spatial_mean_kernel<<<grid, 256, 0, ST(stream)>>>(x, out, HW, C);
  return check_launch("spatial_mean_kernel");
}

int udb_aa_resize_nhwc_f16(const void* in, void* out, int32_t B, int32_t H, int32_t W, int32_t C, int32_t oh, int32_t ow, void* stream) {
  if (C % 8) { set_error("udb_aa_resize_nhwc_f16: C must be a multiple of 8"); return 1; }
  note_work(0.0, 2.0 * B * C * ((double)H * W + (double)oh * ow));
  aa_resize_nhwc_kernel<<<grid_1d((long long)B * oh * ow * (C / 8)), 256, 0, ST(stream)>>>(
      reinterpret_cast<const __half*>(in), reinterpret_cast<__half*>(out), B, H, W, C, oh, ow, (float)H / (float)oh, (float)W / (float)ow);
  return check_launch("aa_resize_nhwc_kernel");
}

int udb_v1_rays_sh81(const udb_v1_rays_t* p, void* stream) {
  const long long toks = (long long)p->B * p->gh * p->gw;
  rays_sh81_kernel<<<(int)((toks + 7) / 8), 256, 0, ST(stream)>>>(*p);
  return check_launch("rays_sh81_kernel");
}

int udb_v1_camera_intrinsics(const float* x4, const float* gt_k, int32_t B, int32_t net_h, int32_t net_w, float ratio, int32_t pad_l,
                             int32_t pad_t, int32_t skip_camera, float* intr4_rays, float* k_out, float* k4_points, void* stream) {
  v1_camera_intrinsics_kernel<<<(B + 63) / 64, 64, 0, ST(stream)>>>(x4, gt_k, B, net_h, net_w, ratio, pad_l, pad_t, skip_camera, intr4_rays, k_out,
                                                                     k4_points);
  return check_launch("v1_camera_intrinsics_kernel");
}

int udb_cross_attn_small(const float* q, const float* q_pos, const void* kv, float* out, float* scratch, int32_t B, int32_t nq, int32_t nk,
                         int32_t D, float scale, void* stream) {
  if (nq < 1 || nq > CA_MAXQ || D % 256 || !scratch) { set_error("udb_cross_attn_small: nq=%d D=%d unsupported (nq <= 4, D %% 256 == 0)", nq, D); return 1; }
  const int chunk = (nk + CA_SPLITS - 1) / CA_SPLITS;
  const size_t smem = (size_t)(nq * D + nq * chunk + 16) * 4;
  if (smem > 200 * 1024) { set_error("udb_cross_attn_small: nk=%d too large", nk); return 1; }
  static std::atomic<size_t> set_for[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (smem > 48 * 1024 && smem > set_for[dev & 63].load()) {
    if (cudaFuncSetAttribute(cross_attn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      set_error("udb_cross_attn_small: cudaFuncSetAttribute failed"); return 1;
    }
    set_for[dev & 63].store(smem);
  }
  note_work(4.0 * B * nq * (double)nk * D, 4.0 * B * nk * D);
  cross_attn_partial_kernel<<<dim3(CA_SPLITS, B), 256, smem, ST(stream)>>>(q, q_pos, reinterpret_cast<const __half*>(kv), scratch, nq, nk, D, scale);
  if (check_launch("cross_attn_partial_kernel")) return 1;
  cross_attn_merge_kernel<<<dim3(nq, B), 256, 0, ST(stream)>>>(scratch, out, nq, D);
  return check_launch("cross_attn_merge_kernel");
}

int udb_softmax_rows(const float* s, void* p, int64_t rows, int32_t n_valid, int32_t ld_in, int32_t ld_out, float scale, void* stream) {
  softmax_rows_kernel<<<(int)((rows + 7) / 8), 256, 0, ST(stream)>>>(s, reinterpret_cast<__half*>(p), rows, n_valid, ld_in, ld_out, scale);
  return check_launch("softmax_rows_kernel");
}

int udb_add_f32(const float* a, const float* b, float* out, void* out_f16, int64_t n, void* stream) {
  if (n % 4) { set_error("udb_add_f32: n must be a multiple of 4"); return 1; }
  note_work(0.0, (8.0 + (out ? 4.0 : 0.0) + (out_f16 ? 2.0 : 0.0)) * n);
  add_f32_kernel<<<grid_1d(n / 4), 256, 0, ST(stream)>>>(reinterpret_cast<const float4*>(a), reinterpret_cast<const float4*>(b),
                                                         reinterpret_cast<float4*>(out), reinterpret_cast<uint2*>(out_f16), n / 4);
  return check_launch("add_f32_kernel");
}

int udb_copy_rows_f32_to_f16(const float* src, void* dst, int32_t groups, int32_t rows_per_group, int32_t D, int64_t dst_group_stride,
                             int64_t dst_row0, void* stream) {
  copy_rows_f16_kernel<<<grid_1d((long long)groups * rows_per_group * D), 256, 0, ST(stream)>>>(src, reinterpret_cast<__half*>(dst), groups,
                                                                                                rows_per_group, D, dst_group_stride, dst_row0);
  return check_launch("copy_rows_f16_kernel");
}

int udb_conv3x3_c1_exp(const void* x, const float* w, float bias, float* out, int32_t B, int32_t H, int32_t W, int32_t C, void* stream) {
  if (C != 64 && C != 128 && C != 256) { set_error("udb_conv3x3_c1_exp: C=%d unsupported (64, 128 or 256)", C); return 1; }
  const long long px = (long long)B * H * W;
  const int lpp = C / 8, ppb = 8 * (32 / lpp);
  const int grid = (int)((px + ppb - 1) / ppb);
  note_work(2.0 * px * 9 * C, 2.0 * px * C + 4.0 * px);
  const __half* xh = reinterpret_cast<const __half*>(x);
  if (lpp == 8) conv3x3_c1_kernel<8><<<grid, 256, 0, ST(stream)>>>(xh, w, bias, out, B, H, W, C);
  else if (lpp == 16) conv3x3_c1_kernel<16><<<grid, 256, 0, ST(stream)>>>(xh, w, bias, out, B, H, W, C);
  else conv3x3_c1_kernel<32><<<grid, 256, 0, ST(stream)>>>(xh, w, bias, out, B, H, W, C);
  return check_launch("conv3x3_c1_kernel");
}

int udb_nystrom_landmarks(const void* q, int32_t ldq, const void* kv, int32_t ldkv, void* out, int32_t B, int32_t n, int32_t heads, void* stream) {
  if (n < 128) { set_error("udb_nystrom_landmarks: sequence %d shorter than the 128 landmarks", n); return 1; }
  nystrom_landmarks_kernel<<<dim3(128, heads, B), 64, 0, ST(stream)>>>(reinterpret_cast<const __half*>(q), ldq, reinterpret_cast<const __half*>(kv),
                                                                       ldkv, reinterpret_cast<__half*>(out), n, heads, 128);
  return check_launch("nystrom_landmarks_kernel");
}

int udb_nystrom_k2_pinv(const void* landmarks, float* k2, float* z, float* tmp, int32_t B, int32_t heads, int32_t iters, void* stream) {
  // kernel_2 = softmax(ql kl^T / 8); Z = pinv(kernel_2) by `iters` Newton-Schulz steps (Razavi et al.):
  //   KV = K Z;  T1 = 7I - KV;  T2 = 15I - KV T1;  T3 = 13I - KV T2;  Z <- 0.25 Z T3        (tmp: 3 matrices per (b, head))
  const int m = 128, nb = B * heads;
  const long long mm = (long long)m * m;
  nystrom_k2_kernel<<<dim3(m / 4, nb), 128, 0, ST(stream)>>>(reinterpret_cast<const __half*>(landmarks), k2, heads, m);
  if (check_launch("nystrom_k2_kernel")) return 1;
  nystrom_pinv_init_kernel<<<nb, 128, 0, ST(stream)>>>(k2, z, m);
  if (check_launch("nystrom_pinv_init_kernel")) return 1;
  float* KV = tmp;
  float* Ta = tmp + nb * mm;
  float* Tb = tmp + 2 * nb * mm;
  auto mmul = [&](const float* A, const float* Bm, float* C, float alpha, float diag) {
    BmmArgs a{};
    a.A = A; a.sA = mm; a.lda = m;
    a.Bp = Bm; a.sB1 = mm; a.sB2 = 0; a.ldb = m; a.b_f16 = 0; a.inner = 1;
    a.C = C; a.sC1 = mm; a.sC2 = 0; a.ldc = m; a.c_f16 = 0;
    a.M = m; a.N = m; a.K = m; a.alpha = alpha; a.diag = diag;
    bmm_f32_kernel<<<dim3(m / 64, m / 64, nb), 256, 0, ST(stream)>>>(a);
    return check_launch("bmm_f32_kernel");
  };
  float* Z = z;
  float* spare = Tb;
  for (int it = 0; it < iters; ++it) {
    float* T2 = spare;
    if (mmul(k2, Z, KV, 1.f, 0.f)) return 1;                       // KV = K Z
    eye_minus_kernel<<<grid_1d(nb * mm), 256, 0, ST(stream)>>>(KV, Ta, 7.f, m, nb * mm);     // T1 = 7I - KV
    if (check_launch("eye_minus_kernel")) return 1;
    if (mmul(KV, Ta, T2, -1.f, 15.f)) return 1;                    // T2 = 15I - KV T1
    if (mmul(KV, T2, Ta, -1.f, 13.f)) return 1;                    // T3 = 13I - KV T2   (over T1)
    if (mmul(Z, Ta, T2, 0.25f, 0.f)) return 1;                     // Z' = 0.25 Z T3     (over T2)
    spare = Z;
    Z = T2;
  }
  if (Z != z && cudaMemcpyAsync(z, Z, sizeof(float) * nb * mm, cudaMemcpyDeviceToDevice, ST(stream)) != cudaSuccess) {
    set_error("udb_nystrom_k2_pinv: copy failed"); return 1;
  }
  return 0;
}

// out[(b, lm), h*64 + d] (f16, row stride ldo) = sum_j Z[b,h][lm][j] * k3[(b, j), h*64 + d]: the (pinv . kernel_3) product that
// becomes the V operand of the final softmax(q kl^T) attention.
int udb_nystrom_zk3(const float* z, const void* k3, int32_t ldk3, void* out, int32_t ldo, int32_t B, int32_t heads, void* stream) {
  const int m = 128;
  BmmArgs a{};
  a.A = z; a.sA = (long long)m * m; a.lda = m;
  a.Bp = k3; a.sB1 = (long long)m * ldk3; a.sB2 = 64; a.ldb = ldk3; a.b_f16 = 1; a.inner = heads;
  a.C = out; a.sC1 = (long long)m * ldo; a.sC2 = 64; a.ldc = ldo; a.c_f16 = 1;
  a.M = m; a.N = 64; a.K = m; a.alpha = 1.f; a.diag = 0.f;
  bmm_f32_kernel<<<dim3(1, m / 64, B * heads), 256, 0, ST(stream)>>>(a);
  return check_launch("bmm_f32_kernel");
}

int udb_v1_mean_maps(const float* o8, const float* o4, const float* o2, float* mean, int32_t B, int32_t gh, int32_t gw, int32_t net_h,
                     int32_t net_w, void* stream) {
  v1_mean_maps_kernel<<<grid_1d((long long)B * net_h * net_w), 256, 0, ST(stream)>>>(o8, o4, o2, mean, B, gh, gw, net_h, net_w);
  return check_launch("v1_mean_maps_kernel");
}

int udb_v1_postprocess(const udb_v1_postprocess_t* p, void* stream) {
  v1_postprocess_kernel<<<grid_1d((long long)p->B * p->H * p->W), 256, 0, ST(stream)>>>(*p);
  return check_launch("v1_postprocess_kernel");
}

}  // extern "C"
