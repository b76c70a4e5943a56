// Bandwidth-bound helper kernels around the tcgen05 convolution (all NHWC fp16 unless noted), sm_100a.
//
// Reference (SipMask-mmdetection/mmdet/):
//   ops/norm.py:43-49 + ops/conv_module.py:124-132            GroupNorm(32) + ReLU after tower convs
//   ops/dcn/src/deform_conv_cuda_kernel.cu:85-115,191-243      deformable im2col (bilinear gather)
//   models/anchor_heads/sipmask_head.py:30-33,49-50            conv_offset 1x1 (4 -> 72, no bias)
//   models/backbones/resnet.py:460                             MaxPool2d(3, 2, 1)
//   models/anchor_heads/sipmask_head.py:279,285                F.interpolate(bilinear, align_corners=False)
//   datasets/pipelines/formating.py ImageToTensor              NCHW fp32 input image
// Every kernel moves 16-byte vectors (8 fp16 channels) per thread so that a warp covers whole 128-byte lines.
#include "common.cuh"

namespace smb {

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 u;
  __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
  return u;
}

// ------------------------------------------------------------------------------------------ GroupNorm
// stats[(img*G + g)*2 + {0,1}] = {sum * 2^20, sum of squares * 2^16} as int64 over hw * (C/G) elements.
__global__ void gn_apply_kernel(__half* __restrict__ x, int n_img, int hw, int C, int pitch, const long long* __restrict__ stats,
                                const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int relu) {
  const int vecs = C >> 3;
  const long long total = (long long)n_img * hw * vecs;
  const int G = 32, cpg = C / G;
  const float inv_cnt = 1.0f / ((float)hw * (float)cpg);
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int v = (int)(t % vecs);
    const unsigned row = t / (unsigned)vecs;
    const int img = (int)(row / hw);
    uint4* p = reinterpret_cast<uint4*>(x + (size_t)row * pitch + v * 8);
    float f[8];
    unpack8(*p, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = v * 8 + j;
      const int g = c / cpg;
      // int64 -> fp32 with ONE rounding; the 2^-20 / 2^-16 scales are exact, so this equals the former double-precision
      // product bit for bit without FP64 instructions (B200 issues those at a small fraction of the fp32 rate)
      const float s = __ll2float_rn(stats[((size_t)img * G + g) * 2]) * (1.0f / kGnSumScale);
      const float ss = __ll2float_rn(stats[((size_t)img * G + g) * 2 + 1]) * (1.0f / kGnSqScale);
      const float mean = s * inv_cnt;
      const float var = fmaxf(ss * inv_cnt - mean * mean, 0.f);
      const float rstd = rsqrtf(var + eps);
      float y = (f[j] - mean) * rstd * gamma[c] + beta[c];
      f[j] = relu ? fmaxf(y, 0.f) : y;
    }
    *p = pack8(f);
  }
}

// One CTA handles `rows_per_cta` pixels of one image; thread -> (row lane, 8-channel vector).
__global__ void gn_stats_kernel(const __half* __restrict__ x, int hw, int C, int pitch, int rows_per_cta,
                                long long* __restrict__ stats) {
  __shared__ unsigned long long s_sum[32], s_sq[32];
  const int img = blockIdx.y;
  const int vecs = C >> 3;
  const int cpg = C / 32;
  if (threadIdx.x < 32) { s_sum[threadIdx.x] = 0ull; s_sq[threadIdx.x] = 0ull; }
  __syncthreads();
  const int v = threadIdx.x % vecs;
  const int rl = threadIdx.x / vecs;
  const int rstep = blockDim.x / vecs;
  const int r0 = blockIdx.x * rows_per_cta;
  const int r1 = min(r0 + rows_per_cta, hw);
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s[j] = 0.f; q[j] = 0.f; }
  if (rl < rstep) {
    for (int r = r0 + rl; r < r1; r += rstep) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + ((size_t)img * hw + r) * pitch + v * 8));
      float f[8];
      unpack8(u, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] += f[j] * f[j]; }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int g = (v * 8 + j) / cpg;
      atomicAdd(&s_sum[g], (unsigned long long)__float2ll_rn(s[j] * kGnSumScale));
      atomicAdd(&s_sq[g], (unsigned long long)__float2ll_rn(q[j] * kGnSqScale));
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    unsigned long long* st = reinterpret_cast<unsigned long long*>(stats);
    atomicAdd(st + ((size_t)img * 32 + threadIdx.x) * 2, s_sum[threadIdx.x]);
    atomicAdd(st + ((size_t)img * 32 + threadIdx.x) * 2 + 1, s_sq[threadIdx.x]);
  }
}

// ------------------------------------------------------------------------- DCN offsets + deformable im2col
// offset[pix, o] = sum_k W[o,k] * (bbox[pix,k] * scale)      (1x1 conv 4 -> dg*18, no bias)
__global__ void offset_conv_kernel(const float* __restrict__ bbox, int bbox_pitch, float scale, const float* __restrict__ w,
                                   int n_off, float* __restrict__ off, long long npix) {
  const long long total = npix * n_off;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int o = (int)(t % n_off);
    const unsigned pix = t / (unsigned)n_off;
    const float* b = bbox + (size_t)pix * bbox_pitch;
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) acc = fmaf(__fmul_rn(b[k], scale), w[o * 4 + k], acc);
    off[t] = acc;
  }
}

// One warp per (pixel, tap): lanes cover the C/8 channel vectors (C <= 256 per pass).
// col[pix, tap*C + c] = bilinear(x[:, :, c], h + i - 1 + dh, w + j - 1 + dw), zero outside (-1,H)x(-1,W)
// with per-corner bounds exactly as deform_conv_cuda_kernel.cu:98-109,229.
__global__ void deform_im2col_kernel(const __half* __restrict__ x, const float* __restrict__ off, int off_pitch,
                                     __half* __restrict__ col, int n_img, int H, int W, int C, int dg) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const long long total = (long long)n_img * H * W * 9;
  const int vecs = C >> 3;
  const int cpg = C / dg;
  for (long long wq = blockIdx.x * (long long)warps_per_block + (threadIdx.x >> 5); wq < total;
       wq += (long long)gridDim.x * warps_per_block) {
    const int tap = (int)(wq % 9);
    const long long pix = wq / 9;
    const int w_ = (int)(pix % W);
    const int h_ = (int)((pix / W) % H);
    const int img = (int)(pix / ((long long)W * H));
    const int i = tap / 3, j = tap - i * 3;
    const __half* xim = x + (size_t)img * H * W * C;
    for (int v = lane; v < vecs; v += 32) {
      const int g = (v * 8) / cpg;
      const float* o = off + pix * off_pitch + g * 18 + 2 * tap;
      const float h_im = (float)(h_ - 1 + i) + o[0];
      const float w_im = (float)(w_ - 1 + j) + o[1];
      float r[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) r[e] = 0.f;
      if (h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W) {
        const int h_low = (int)floorf(h_im), w_low = (int)floorf(w_im);
        const int h_high = h_low + 1, w_high = w_low + 1;
        const float lh = h_im - (float)h_low, lw = w_im - (float)w_low;
        const float hh = 1.f - lh, hw = 1.f - lw;
        const float w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
        float f[8];
        if (h_low >= 0 && w_low >= 0) {
          unpack8(__ldg(reinterpret_cast<const uint4*>(xim + ((size_t)h_low * W + w_low) * C + v * 8)), f);
#pragma unroll
          for (int e = 0; e < 8; ++e) r[e] = w1 * f[e];
        }
        if (h_low >= 0 && w_high <= W - 1) {
          unpack8(__ldg(reinterpret_cast<const uint4*>(xim + ((size_t)h_low * W + w_high) * C + v * 8)), f);
#pragma unroll
          for (int e = 0; e < 8; ++e) r[e] += w2 * f[e];
        }
        if (h_high <= H - 1 && w_low >= 0) {
          unpack8(__ldg(reinterpret_cast<const uint4*>(xim + ((size_t)h_high * W + w_low) * C + v * 8)), f);
#pragma unroll
          for (int e = 0; e < 8; ++e) r[e] += w3 * f[e];
        }
        if (h_high <= H - 1 && w_high <= W - 1) {
          unpack8(__ldg(reinterpret_cast<const uint4*>(xim + ((size_t)h_high * W + w_high) * C + v * 8)), f);
#pragma unroll
          for (int e = 0; e < 8; ++e) r[e] += w4 * f[e];
        }
      }
      *reinterpret_cast<uint4*>(col + (size_t)pix * 9 * C + (size_t)tap * C + v * 8) = pack8(r);
    }
  }
}

// -------------------------------------------------------------------------------------------- max pool
__global__ void maxpool3x3s2_kernel(const __half* __restrict__ x, __half* __restrict__ y, int N, int H, int W, int C, int Ho,
                                    int Wo) {
  pdl_wait();
  const int vecs = C >> 3;
  const long long total = (long long)N * Ho * Wo * vecs;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int v = (int)(t % vecs);
    unsigned q = t / (unsigned)vecs;
    const int ox = (int)(q % Wo); q /= Wo;
    const int oy = (int)(q % Ho);
    const int n = (int)(q / Ho);
    float m[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) m[e] = -INFINITY;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      const int iy = oy * 2 - 1 + dy;
      if (iy < 0 || iy >= H) continue;
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int ix = ox * 2 - 1 + dx;
        if (ix < 0 || ix >= W) continue;
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(x + (((size_t)n * H + iy) * W + ix) * C + v * 8)), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) m[e] = fmaxf(m[e], f[e]);
      }
    }
    *reinterpret_cast<uint4*>(y + (((size_t)n * Ho + oy) * Wo + ox) * C + v * 8) = pack8(m);
  }
}

// ------------------------------------------------------------------------------------ bilinear upsample
// PyTorch upsample_bilinear2d, align_corners=False, scale_factor = factor (integer):
//   src = max((dst + 0.5) / factor - 0.5, 0); i0 = (int)src; i1 = i0 + (i0 < in-1); l1 = src - i0
// y is [N, Ho, Wo, out_pitch] with Ho <= H * factor, Wo <= W * factor: the top-left Ho x Wo of the upsampled map.
__global__ void upsample_bilinear_kernel(const __half* __restrict__ x, int in_pitch, __half* __restrict__ y, int out_pitch,
                                         int out_choff, int N, int H, int W, int C, int factor, int Ho, int Wo, int relu) {
  pdl_wait();
  const int vecs = C >> 3;
  const float rs = 1.0f / (float)factor;
  const long long total = (long long)N * Ho * Wo * vecs;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int v = (int)(t % vecs);
    unsigned q = t / (unsigned)vecs;
    const int ox = (int)(q % Wo); q /= Wo;
    const int oy = (int)(q % Ho);
    const int n = (int)(q / Ho);
    float sy = ((float)oy + 0.5f) * rs - 0.5f; sy = sy < 0.f ? 0.f : sy;
    float sx = ((float)ox + 0.5f) * rs - 0.5f; sx = sx < 0.f ? 0.f : sx;
    const int y0 = (int)sy, x0 = (int)sx;
    const int y1 = y0 + (y0 < H - 1 ? 1 : 0), x1 = x0 + (x0 < W - 1 ? 1 : 0);
    const float ly = sy - (float)y0, lx = sx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    const __half* b = x + (size_t)n * H * W * in_pitch + v * 8;
    float f00[8], f01[8], f10[8], f11[8], r[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(b + ((size_t)y0 * W + x0) * in_pitch)), f00);
    unpack8(__ldg(reinterpret_cast<const uint4*>(b + ((size_t)y0 * W + x1) * in_pitch)), f01);
    unpack8(__ldg(reinterpret_cast<const uint4*>(b + ((size_t)y1 * W + x0) * in_pitch)), f10);
    unpack8(__ldg(reinterpret_cast<const uint4*>(b + ((size_t)y1 * W + x1) * in_pitch)), f11);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float val = hy * (hx * f00[e] + lx * f01[e]) + ly * (hx * f10[e] + lx * f11[e]);
      r[e] = relu ? fmaxf(val, 0.f) : val;
    }
    *reinterpret_cast<uint4*>(y + (((size_t)n * Ho + oy) * Wo + ox) * out_pitch + out_choff + v * 8) = pack8(r);
  }
}

// plain strided copy of a channel block (level 0 of the prototype concat: torch.cat is a copy in the reference)
__global__ void copy_channels_kernel(const __half* __restrict__ x, int in_pitch, __half* __restrict__ y, int out_pitch,
                                     int out_choff, long long npix, int C, int relu) {
  pdl_wait();
  const int vecs = C >> 3;
  const long long total = npix * vecs;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int v = (int)(t % vecs);
    const unsigned pix = t / (unsigned)vecs;
    uint4 u = __ldg(reinterpret_cast<const uint4*>(x + (size_t)pix * in_pitch + v * 8));
    if (relu) {
      __half2* h = reinterpret_cast<__half2*>(&u);
      const __half2 z = __float2half2_rn(0.f);
#pragma unroll
      for (int i = 0; i < 4; ++i) h[i] = __hmax2(h[i], z);
    }
    *reinterpret_cast<uint4*>(y + (size_t)pix * out_pitch + out_choff + v * 8) = u;
  }
}

// --------------------------------------------------------------------------------------- image -> NHWC8
// img [N,3,H,W] fp32 -> out [N, H+6, W+8, 8] fp16, pixel (y,x) at (y+3, x+3), zeros elsewhere / in ch 3..7.
__global__ void image_to_nhwc8_kernel(const float* __restrict__ img, __half* __restrict__ out, int N, int H, int W) {
  pdl_wait();
  const int Hp = H + 6, Wp = W + 8;
  const long long total = (long long)N * Hp * Wp;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int xp = (int)(t % Wp);
    const int yp = (int)((t / Wp) % Hp);
    const int n = (int)(t / ((long long)Wp * Hp));
    const int x = xp - 3, y = yp - 3;
    float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (x >= 0 && x < W && y >= 0 && y < H) {
      const size_t plane = (size_t)H * W;
      const float* p = img + (size_t)n * 3 * plane + (size_t)y * W + x;
      f[0] = p[0]; f[1] = p[plane]; f[2] = p[2 * plane];
    }
    *reinterpret_cast<uint4*>(out + (size_t)t * 8) = pack8(f);
  }
}

// img [N,3,H,W] fp32 -> out [N, H/2+3, W/2+4, 16] fp16: the stem's space-to-depth layout, element (Y, X, (dy*2+dx)*4 + c) =
// image pixel (2Y+dy-3, 2X+dx-3), channel c; zeros outside the image and in c == 3.
__global__ void image_to_s2d16_kernel(const float* __restrict__ img, __half* __restrict__ out, int N, int H, int W) {
  pdl_wait();
  const int Hq = H / 2 + 3, Wq = W / 2 + 4;
  const long long total = (long long)N * Hq * Wq;
  const size_t plane = (size_t)H * W;
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int X = (int)(t % Wq);
    const int Y = (int)((t / Wq) % Hq);
    const int n = (int)(t / ((long long)Wq * Hq));
    float f[16];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const int x = 2 * X + (d & 1) - 3, y = 2 * Y + (d >> 1) - 3;
      f[4 * d] = f[4 * d + 1] = f[4 * d + 2] = f[4 * d + 3] = 0.f;
      if (x >= 0 && x < W && y >= 0 && y < H) {
        const float* p = img + (size_t)n * 3 * plane + (size_t)y * W + x;
        f[4 * d] = p[0]; f[4 * d + 1] = p[plane]; f[4 * d + 2] = p[2 * plane];
      }
    }
    uint4* o = reinterpret_cast<uint4*>(out + (size_t)t * 16);
    o[0] = pack8(f);
    o[1] = pack8(f + 8);
  }
}

// ------------------------------------------------------------------------------- multi-level (batched) variants
// The FCOS towers run on five pyramid levels with shared weights; these kernels process all levels in one launch.
constexpr int kMaxLv = 5;
struct MultiDesc {
  int num;
  long long start[kMaxLv + 1];      // prefix of work items per level
  const void* a[kMaxLv];
  const void* b[kMaxLv];
  void* c[kMaxLv];
  int H[kMaxLv], W[kMaxLv];
  float scale[kMaxLv];
};

__device__ __forceinline__ int find_level(const MultiDesc& d, long long t) {
  int l = 0;
#pragma unroll
  for (int i = 1; i < kMaxLv; ++i)
    if (i < d.num && t >= d.start[i]) l = i;
  return l;
}

// GroupNorm(32) + ReLU in place; a[l] = x (fp16 [n_img*hw, C]), b[l] = stats (int64 fixed point).  C/32 % 8 == 0.
__global__ void gn_apply_multi_kernel(MultiDesc d, int n_img, int C, int pitch, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, float eps, int relu) {
  pdl_wait();
  const int vecs = C >> 3;
  const int cpg = C / 32;
  const long long total = d.start[d.num];
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int l = find_level(d, t);
    const unsigned q = t - (unsigned)d.start[l];
    const int hw = d.H[l] * d.W[l];
    const int v = (int)(q % vecs);
    const unsigned row = q / (unsigned)vecs;
    const int img = (int)(row / hw);
    const int g = (v * 8) / cpg;
    const long long* st = reinterpret_cast<const long long*>(d.b[l]) + ((size_t)img * 32 + g) * 2;
    const float inv_cnt = 1.0f / ((float)hw * (float)cpg);
    // int64 -> fp32 with one rounding, exact power-of-two scales: same bits as the double-precision product, no FP64 issue
    const float mean = __ll2float_rn(st[0]) * (1.0f / kGnSumScale) * inv_cnt;
    const float ex2 = __ll2float_rn(st[1]) * (1.0f / kGnSqScale) * inv_cnt;
    const float rstd = rsqrtf(fmaxf(ex2 - mean * mean, 0.f) + eps);
    uint4* p = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(d.c[l]) + (size_t)row * pitch + v * 8);
    float f[8];
    unpack8(*p, f);
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8) + 1);
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + v * 8)), b1 = __ldg(reinterpret_cast<const float4*>(beta + v * 8) + 1);
    const float ga[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    const float be[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float y = (f[j] - mean) * rstd * ga[j] + be[j];
      f[j] = relu ? fmaxf(y, 0.f) : y;
    }
    *p = pack8(f);
  }
}

// Same arithmetic, thread-stationary in the channel vector: a CTA owns kGnRows consecutive pixel rows of ONE (level, image),
// a thread one 8-channel vector (v = tid % vecs) of every (256 / vecs)-th of those rows.  Level lookup, statistics (two
// int64 loads, conversions, rsqrt) and gamma / beta (four 16-byte loads) are evaluated once per thread instead of once per
// 16-byte vector (gn_apply_multi_kernel: ~150 instructions per vector, 67 % issue-bound at 10 us for 23 MB in the r02 ncu
// capture); the row loop is a load, 8 x (sub, mul, fma, max), a store.  start[] holds the prefix of CTAs per level.
constexpr int kGnRows = 64;
__global__ void __launch_bounds__(256) gn_apply_rows_kernel(MultiDesc d, int n_img, int C, int pitch, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps, int relu) {
  pdl_wait();
  const int vecs = C >> 3;                                   // 256 % vecs == 0 (host-checked)
  const int cpg = C / 32;
  const int l = find_level(d, (long long)blockIdx.x);
  const int q = (int)blockIdx.x - (int)d.start[l];
  const int hw = d.H[l] * d.W[l];
  const int per_img = (hw + kGnRows - 1) / kGnRows;          // CTAs per image of this level
  const int img = q / per_img;
  const int r0 = (q - img * per_img) * kGnRows, r1 = min(hw, r0 + kGnRows);
  const int v = (int)threadIdx.x % vecs, rsub = (int)threadIdx.x / vecs, rstep = 256 / vecs;
  const int g = (v * 8) / cpg;
  const long long* st = reinterpret_cast<const long long*>(d.b[l]) + ((size_t)img * 32 + g) * 2;
  const float inv_cnt = 1.0f / ((float)hw * (float)cpg);
  const float mean = __ll2float_rn(st[0]) * (1.0f / kGnSumScale) * inv_cnt;
  const float ex2 = __ll2float_rn(st[1]) * (1.0f / kGnSqScale) * inv_cnt;
  const float rstd = rsqrtf(fmaxf(ex2 - mean * mean, 0.f) + eps);
  const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8) + 1);
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + v * 8)), b1 = __ldg(reinterpret_cast<const float4*>(beta + v * 8) + 1);
  const float ga[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
  const float be[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
  __half* base = reinterpret_cast<__half*>(d.c[l]) + (size_t)img * hw * pitch + v * 8;
#pragma unroll 4
  for (int r = r0 + rsub; r < r1; r += rstep) {
    uint4* p = reinterpret_cast<uint4*>(base + (size_t)r * pitch);
    float f[8];
    unpack8(*p, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float y = (f[j] - mean) * rstd * ga[j] + be[j];   // the expression of gn_apply_multi_kernel: same bits
      f[j] = relu ? fmaxf(y, 0.f) : y;
    }
    *p = pack8(f);
  }
}

// offsets for all levels: a[l] = raw fcos_reg (fp32, pitch bbox_pitch), c[l] = offsets fp32 [hw, n_off], scale[l] = Scale_l
__global__ void offset_conv_multi_kernel(MultiDesc d, int bbox_pitch, const float* __restrict__ w, int n_off) {
  pdl_wait();
  const long long total = d.start[d.num];
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)total; t += blockDim.x * gridDim.x) {   // 32-bit index math: 64-bit div/mod costs ~100 instructions each
    const int l = find_level(d, t);
    const unsigned q = t - (unsigned)d.start[l];
    const int o = (int)(q % n_off);
    const unsigned pix = q / (unsigned)n_off;
    const float* b = reinterpret_cast<const float*>(d.a[l]) + (size_t)pix * bbox_pitch;
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) acc = fmaf(__fmul_rn(b[k], d.scale[l]), w[o * 4 + k], acc);
    reinterpret_cast<float*>(d.c[l])[q] = acc;
  }
}

// deformable im2col for all levels: a[l] = x fp16 [n,H,W,C], b[l] = offsets fp32 [n,H,W,dg*18], c[l] = col fp16 [n,H,W,9C]
// work item = one pixel handled by one warp: all 9 taps x 4 bilinear corners are independent 16-byte loads (36 in
// flight per lane), the offsets of a pixel are read once, index math is 32-bit.
__global__ void __launch_bounds__(256) deform_im2col_multi_kernel(MultiDesc d, int off_pitch, int C, int dg) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const int total = (int)d.start[d.num];          // pixels over all levels (items_per_pixel == 1)
  const int vecs = C >> 3;
  const int cpg = C / dg;
  for (int wq0 = blockIdx.x * warps_per_block + (threadIdx.x >> 5); wq0 < total; wq0 += gridDim.x * warps_per_block) {
    int l = 0;
#pragma unroll
    for (int i = 1; i < kMaxLv; ++i)
      if (i < d.num && wq0 >= (int)d.start[i]) l = i;
    const int pix = wq0 - (int)d.start[l];
    const int H = d.H[l], W = d.W[l];
    const int w_ = pix % W;
    const int hq = pix / W;
    const int h_ = hq % H;
    const int img = hq / H;
    const __half* xim = reinterpret_cast<const __half*>(d.a[l]) + (size_t)img * H * W * C;
    const float* off = reinterpret_cast<const float*>(d.b[l]) + (size_t)pix * off_pitch;
    __half* col = reinterpret_cast<__half*>(d.c[l]) + (size_t)pix * 9 * C;
    for (int v = lane; v < vecs; v += 32) {
      const int g = (v * 8) / cpg;
      const float* og = off + g * 18;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int i = tap / 3, j = tap - i * 3;
        const float h_im = (float)(h_ - 1 + i) + og[2 * tap];
        const float w_im = (float)(w_ - 1 + j) + og[2 * tap + 1];
        float r[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) r[e] = 0.f;
        if (h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W) {
          const int h_low = (int)floorf(h_im), w_low = (int)floorf(w_im);
          const int h_high = h_low + 1, w_high = w_low + 1;
          const float lh = h_im - (float)h_low, lw = w_im - (float)w_low;
          const float hh = 1.f - lh, hw = 1.f - lw;
          const float w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
          const bool ok1 = h_low >= 0 && w_low >= 0, ok2 = h_low >= 0 && w_high <= W - 1;
          const bool ok3 = h_high <= H - 1 && w_low >= 0, ok4 = h_high <= H - 1 && w_high <= W - 1;
          const uint4 z = make_uint4(0u, 0u, 0u, 0u);
          const uint4 u1 = ok1 ? __ldg(reinterpret_cast<const uint4*>(xim + (h_low * W + w_low) * C + v * 8)) : z;
          const uint4 u2 = ok2 ? __ldg(reinterpret_cast<const uint4*>(xim + (h_low * W + w_high) * C + v * 8)) : z;
          const uint4 u3 = ok3 ? __ldg(reinterpret_cast<const uint4*>(xim + (h_high * W + w_low) * C + v * 8)) : z;
          const uint4 u4 = ok4 ? __ldg(reinterpret_cast<const uint4*>(xim + (h_high * W + w_high) * C + v * 8)) : z;
          float f1[8], f2[8], f3[8], f4[8];
          unpack8(u1, f1); unpack8(u2, f2); unpack8(u3, f3); unpack8(u4, f4);
#pragma unroll
          for (int e = 0; e < 8; ++e) r[e] = (w1 * f1[e] + w2 * f2[e] + w3 * f3[e] + w4 * f4[e]);
        }
        *reinterpret_cast<uint4*>(col + tap * C + v * 8) = pack8(r);
      }
    }
  }
}

static inline int grid_for(long long total, int block) {
  // the grid-stride kernels index their work items with 32 bits (64-bit div / mod costs ~100 instructions each on the GPU);
  // 2^31 items = 16 GB of fp16 vectors, far beyond any tensor on this path
  if (total >= (1LL << 31)) { fprintf(stderr, "sipmask_b200: %lld work items exceed the 32-bit index range\n", total); abort(); }
  long long g = (total + block - 1) / block;
  const long long cap = 148LL * 32;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace smb

using namespace smb;

extern "C" int smb_groupnorm_relu_apply(void* x, int n_img, int hw, int C, int pitch, const void* stats, const float* gamma,
                                        const float* beta, float eps, int relu, smb_stream_t stream) {
  SMB_CHECK_ARG(x && stats && gamma && beta, "smb_groupnorm_relu_apply: null pointer");
  SMB_CHECK_ARG(C % 32 == 0 && C % 8 == 0 && pitch % 8 == 0 && hw > 0 && n_img > 0, "smb_groupnorm_relu_apply: bad shape");
  const long long total = (long long)n_img * hw * (C / 8);
  gn_apply_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((__half*)x, n_img, hw, C, pitch, (const long long*)stats, gamma, beta,
                                                                          eps, relu);
  SMB_LAUNCH_OK("gn_apply_kernel");
  return SMB_OK;
}

extern "C" int smb_groupnorm_stats(const void* x, int n_img, int hw, int C, int pitch, void* stats, smb_stream_t stream) {
  SMB_CHECK_ARG(x && stats, "smb_groupnorm_stats: null pointer");
  SMB_CHECK_ARG(C % 32 == 0 && C % 8 == 0 && C <= 2048 && pitch % 8 == 0 && hw > 0 && n_img > 0, "smb_groupnorm_stats: bad shape");
  SMB_CUDA_OK(cudaMemsetAsync(stats, 0, sizeof(long long) * n_img * 64, (cudaStream_t)stream));
  const int rows_per_cta = 64;
  dim3 grid(cdiv(hw, rows_per_cta), n_img);
  gn_stats_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __half*)x, hw, C, pitch, rows_per_cta, (long long*)stats);
  SMB_LAUNCH_OK("gn_stats_kernel");
  return SMB_OK;
}

extern "C" int smb_offset_conv1x1(const float* bbox, int bbox_pitch, float scale, const float* weight, int n_off, float* off,
                                  long long npix, smb_stream_t stream) {
  SMB_CHECK_ARG(bbox && weight && off && npix > 0 && n_off > 0, "smb_offset_conv1x1: bad argument");
  offset_conv_kernel<<<grid_for(npix * n_off, 256), 256, 0, (cudaStream_t)stream>>>(bbox, bbox_pitch, scale, weight, n_off, off,
                                                                                    npix);
  SMB_LAUNCH_OK("offset_conv_kernel");
  return SMB_OK;
}

extern "C" int smb_deform_im2col(const void* x, const float* offset, int off_pitch, void* col, int n_img, int H, int W, int C,
                                 int deformable_groups, smb_stream_t stream) {
  SMB_CHECK_ARG(x && offset && col, "smb_deform_im2col: null pointer");
  SMB_CHECK_ARG(C % 8 == 0 && deformable_groups > 0 && C % deformable_groups == 0 && (C / deformable_groups) % 8 == 0,
                "smb_deform_im2col: C=%d dg=%d unsupported", C, deformable_groups);
  const long long warps = (long long)n_img * H * W * 9;
  deform_im2col_kernel<<<grid_for(warps * 32, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)x, offset, off_pitch,
                                                                                    (__half*)col, n_img, H, W, C,
                                                                                    deformable_groups);
  SMB_LAUNCH_OK("deform_im2col_kernel");
  return SMB_OK;
}

extern "C" int smb_maxpool3x3s2(const void* x, void* y, int N, int H, int W, int C, smb_stream_t stream) {
  SMB_CHECK_ARG(x && y && C % 8 == 0, "smb_maxpool3x3s2: bad argument");
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  const long long total = (long long)N * Ho * Wo * (C / 8);
  SMB_CUDA_OK(launch_pdl(maxpool3x3s2_kernel, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)stream, (const __half*)x,
                         (__half*)y, N, H, W, C, Ho, Wo));
  SMB_LAUNCH_OK("maxpool3x3s2_kernel");
  return SMB_OK;
}

extern "C" int smb_upsample_bilinear(const void* x, int in_pitch, void* y, int out_pitch, int out_choff, int N, int H, int W,
                                     int C, int factor, int out_h, int out_w, int relu, smb_stream_t stream) {
  SMB_CHECK_ARG(x && y && C % 8 == 0 && in_pitch % 8 == 0 && out_pitch % 8 == 0 && out_choff % 8 == 0 && factor >= 1 &&
                out_h >= 1 && out_w >= 1 && out_h <= H * factor && out_w <= W * factor &&
                (factor > 1 || (out_h == H && out_w == W)), "smb_upsample_bilinear: bad argument");
  if (factor == 1) {
    const long long npix = (long long)N * H * W;
    SMB_CUDA_OK(launch_pdl(copy_channels_kernel, dim3(grid_for(npix * (C / 8), 256)), dim3(256), 0, (cudaStream_t)stream,
                           (const __half*)x, in_pitch, (__half*)y, out_pitch, out_choff, npix, C, relu));
    SMB_LAUNCH_OK("copy_channels_kernel");
    return SMB_OK;
  }
  const long long total = (long long)N * out_h * out_w * (C / 8);
  SMB_CUDA_OK(launch_pdl(upsample_bilinear_kernel, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)stream, (const __half*)x,
                         in_pitch, (__half*)y, out_pitch, out_choff, N, H, W, C, factor, out_h, out_w, relu));
  SMB_LAUNCH_OK("upsample_bilinear_kernel");
  return SMB_OK;
}

extern "C" int smb_image_to_nhwc8(const float* img, void* out, int N, int H, int W, smb_stream_t stream) {
  SMB_CHECK_ARG(img && out && N > 0 && H > 0 && W > 0, "smb_image_to_nhwc8: bad argument");
  const long long total = (long long)N * (H + 6) * (W + 8);
  SMB_CUDA_OK(launch_pdl(image_to_nhwc8_kernel, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)stream, img, (__half*)out, N,
                         H, W));
  SMB_LAUNCH_OK("image_to_nhwc8_kernel");
  return SMB_OK;
}


// ------------------------------------------------------------------------------------------ multi-level C ABI
static int fill_multi(MultiDesc* d, int num, const int* Hs, const int* Ws, long long items_per_pixel, int n_img) {
  if (num < 1 || num > kMaxLv) return -1;
  d->num = num;
  d->start[0] = 0;
  for (int l = 0; l < num; ++l) {
    if (Hs[l] <= 0 || Ws[l] <= 0) return -1;
    d->H[l] = Hs[l]; d->W[l] = Ws[l];
    d->start[l + 1] = d->start[l] + (long long)n_img * Hs[l] * Ws[l] * items_per_pixel;
  }
  return 0;
}

extern "C" int smb_image_to_s2d16(const float* img, void* out, int N, int H, int W, smb_stream_t stream) {
  SMB_CHECK_ARG(img && out && N > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "smb_image_to_s2d16: bad argument");
  const long long total = (long long)N * (H / 2 + 3) * (W / 2 + 4);
  SMB_CUDA_OK(launch_pdl(image_to_s2d16_kernel, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)stream, img, (__half*)out, N, H, W));
  SMB_LAUNCH_OK("image_to_s2d16_kernel");
  return SMB_OK;
}

extern "C" int smb_groupnorm_relu_apply_multi(int num_levels, void* const* xs, const void* const* stats, const int* Hs,
                                              const int* Ws, int n_img, int C, int pitch, const float* gamma,
                                              const float* beta, float eps, int relu, smb_stream_t stream) {
  SMB_CHECK_ARG(xs && stats && Hs && Ws && gamma && beta, "smb_groupnorm_relu_apply_multi: null pointer");
  SMB_CHECK_ARG(C % 256 == 0 && pitch % 8 == 0 && n_img > 0, "smb_groupnorm_relu_apply_multi: C must be a multiple of 256");
  MultiDesc d;
  SMB_CHECK_ARG(fill_multi(&d, num_levels, Hs, Ws, C / 8, n_img) == 0, "smb_groupnorm_relu_apply_multi: bad levels");
  for (int l = 0; l < num_levels; ++l) { d.c[l] = xs[l]; d.b[l] = stats[l]; d.a[l] = nullptr; d.scale[l] = 1.f; }
  static int rows_kernel = -1;                               // SMB_GN_ROWS=0 keeps the one-vector-per-thread kernel
  if (rows_kernel < 0) { const char* e = getenv("SMB_GN_ROWS"); rows_kernel = e ? atoi(e) : 1; }
  const int vecs = C / 8;
  if (rows_kernel && vecs <= 256 && 256 % vecs == 0) {
    long long ctas = 0;
    for (int l = 0; l < num_levels; ++l) {                   // start[] = prefix of CTAs: n_img * ceil(hw / kGnRows) per level
      d.start[l] = ctas;
      ctas += (long long)n_img * (((long long)Hs[l] * Ws[l] + kGnRows - 1) / kGnRows);
    }
    d.start[num_levels] = ctas;
    SMB_CHECK_ARG(ctas < (1LL << 31), "smb_groupnorm_relu_apply_multi: too many rows");
    SMB_CUDA_OK(launch_pdl(gn_apply_rows_kernel, dim3((unsigned)ctas), dim3(256), 0, (cudaStream_t)stream, d, n_img, C, pitch, gamma,
                           beta, eps, relu));
    SMB_LAUNCH_OK("gn_apply_rows_kernel");
    return SMB_OK;
  }
  SMB_CUDA_OK(launch_pdl(gn_apply_multi_kernel, dim3(grid_for(d.start[num_levels], 256)), dim3(256), 0, (cudaStream_t)stream, d, n_img, C,
                         pitch, gamma, beta, eps, relu));
  SMB_LAUNCH_OK("gn_apply_multi_kernel");
  return SMB_OK;
}

extern "C" int smb_offset_conv1x1_multi(int num_levels, const float* const* bboxes, int bbox_pitch, const float* scales,
                                        const float* weight, int n_off, float* const* offs, const int* Hs, const int* Ws,
                                        int n_img, smb_stream_t stream) {
  SMB_CHECK_ARG(bboxes && scales && weight && offs && Hs && Ws && n_off > 0, "smb_offset_conv1x1_multi: bad argument");
  MultiDesc d;
  SMB_CHECK_ARG(fill_multi(&d, num_levels, Hs, Ws, n_off, n_img) == 0, "smb_offset_conv1x1_multi: bad levels");
  for (int l = 0; l < num_levels; ++l) { d.a[l] = bboxes[l]; d.c[l] = offs[l]; d.b[l] = nullptr; d.scale[l] = scales[l]; }
  SMB_CUDA_OK(launch_pdl(offset_conv_multi_kernel, dim3(grid_for(d.start[num_levels], 256)), dim3(256), 0, (cudaStream_t)stream, d,
                         bbox_pitch, weight, n_off));
  SMB_LAUNCH_OK("offset_conv_multi_kernel");
  return SMB_OK;
}

extern "C" int smb_deform_im2col_multi(int num_levels, const void* const* xs, const float* const* offs, int off_pitch,
                                       void* const* cols, const int* Hs, const int* Ws, int n_img, int C,
                                       int deformable_groups, smb_stream_t stream) {
  SMB_CHECK_ARG(xs && offs && cols && Hs && Ws, "smb_deform_im2col_multi: null pointer");
  SMB_CHECK_ARG(C % 8 == 0 && deformable_groups > 0 && C % deformable_groups == 0 && (C / deformable_groups) % 8 == 0,
                "smb_deform_im2col_multi: C=%d dg=%d unsupported", C, deformable_groups);
  MultiDesc d;
  SMB_CHECK_ARG(fill_multi(&d, num_levels, Hs, Ws, 1, n_img) == 0, "smb_deform_im2col_multi: bad levels");
  for (int l = 0; l < num_levels; ++l) { d.a[l] = xs[l]; d.b[l] = offs[l]; d.c[l] = cols[l]; d.scale[l] = 1.f; }
  SMB_CUDA_OK(launch_pdl(deform_im2col_multi_kernel, dim3(grid_for(d.start[num_levels] * 32, 256)), dim3(256), 0, (cudaStream_t)stream,
                         d, off_pitch, C, deformable_groups));
  SMB_LAUNCH_OK("deform_im2col_multi_kernel");
  return SMB_OK;
}
