// Backward of the small layers around the backbone convolutions (SURVEY.md §8 f1):
//   * MaxPool2d(3, 2, 1) backward                         (autograd of src/resnet.py:141,202)
//   * zero insertion (x2) -- turns the data gradient of a stride-2 conv into a stride-1 conv over a dilated grid
//   * head backward: bilinear-upsample(align_corners) backward restricted to the K live channels, then the backward
//     of the K-row 1x1 scoring conv                       (autograd of src/resnet_dilated.py:27, src/resnet.py:215)
//   * stem weight gradient (7x7 s2, Cin=3): CUDA-core kernel, the K dimension (147) is too thin for TMA im2col
// All deterministic (gather formulations / fixed-order partial sums; no atomics).
#include <stdlib.h>

#include "hk_common.cuh"

namespace hk {

__device__ __forceinline__ void ld8(const __nv_bfloat16* p, float (&f)[8]) {
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  unpack_bf16x2(u.x, f[0], f[1]);
  unpack_bf16x2(u.y, f[2], f[3]);
  unpack_bf16x2(u.z, f[4], f[5]);
  unpack_bf16x2(u.w, f[6], f[7]);
}
__device__ __forceinline__ void st8(__nv_bfloat16* p, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

// ---------------------------------------------------------------- maxpool backward (two deterministic passes)
// pass 1: idx[b,oy,ox,c] = tap (r*3+s) of the first maximum of the window in (r, s) scan order among in-bounds taps -- the element
//         ATen's max_pool2d_with_indices routes the gradient to;
// pass 2: dx[b,iy,ix,c] = sum over the (<= 4) windows containing (iy,ix) of dout[window] * [idx[window] == my tap]   (gather).
// ymax != nullptr: also store the window maxima, i.e. this IS the forward max-pool of the training step (one pass over the stem map
// instead of a forward pass plus this one in the backward).
__global__ void __launch_bounds__(256) maxpool_argmax_kernel(const __nv_bfloat16* __restrict__ x, uint8_t* __restrict__ idx, int B, int H, int W,
                                                            int C, int Ho, int Wo, __nv_bfloat16* __restrict__ ymax = nullptr) {
  const int CG = C >> 3;
  const long long total = (long long)B * Ho * Wo * CG;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % CG);
    long long p = i / CG;
    const int ox = (int)(p % Wo);
    p /= Wo;
    const int oy = (int)(p % Ho);
    const int b = (int)(p / Ho);
    float best[8];
    int who[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { best[j] = -INFINITY; who[j] = -1; }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int yy = 2 * oy - 1 + r;
      if (yy < 0 || yy >= H) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int xx = 2 * ox - 1 + s;
        if (xx < 0 || xx >= W) continue;
        float v[8];
        ld8(x + (((long long)b * H + yy) * W + xx) * C + cg * 8, v);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (v[j] > best[j] || who[j] < 0) { best[j] = v[j]; who[j] = r * 3 + s; }
      }
    }
    uint2 packed;
    packed.x = (uint32_t)who[0] | ((uint32_t)who[1] << 8) | ((uint32_t)who[2] << 16) | ((uint32_t)who[3] << 24);
    packed.y = (uint32_t)who[4] | ((uint32_t)who[5] << 8) | ((uint32_t)who[6] << 16) | ((uint32_t)who[7] << 24);
    *reinterpret_cast<uint2*>(idx + i * 8) = packed;
    if (ymax) st8(ymax + i * 8, best);
  }
}
// One thread per 2x2 block of input pixels (rows 2a, 2a+1; columns 2q, 2q+1) and 8 channels: the four pixels lie in the same four windows
// (oy in {a, a+1}, ox in {q, q+1}), so one index word and one gradient vector per window serve nine (pixel, window) pairs -- 1 window
// read per pixel instead of 2.25 in the one-thread-per-pixel form -- and every pixel's sum still runs over its windows in (oy, ox) order.
__global__ void __launch_bounds__(256) maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ dout, const uint8_t* __restrict__ idx,
                                                         __nv_bfloat16* __restrict__ dx, int B, int H, int W, int C, int Ho, int Wo) {
  const int CG = C >> 3, Hq = (H + 1) >> 1, Wq = (W + 1) >> 1;
  const long long total = (long long)B * Hq * Wq * CG;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % CG);
    long long p = i / CG;
    const int q = (int)(p % Wq);
    p /= Wq;
    const int a = (int)(p % Hq);
    const int b = (int)(p / Hq);
    // window (a + wy, q + wx), wy, wx in {0, 1}
    uint2 w8[2][2];
    uint4 g4[2][2];
#pragma unroll
    for (int wy = 0; wy < 2; ++wy) {
#pragma unroll
      for (int wx = 0; wx < 2; ++wx) {
        const bool live = a + wy < Ho && q + wx < Wo;
        const long long o = (((long long)b * Ho + (a + wy)) * Wo + (q + wx)) * C + cg * 8;
        w8[wy][wx] = live ? __ldg(reinterpret_cast<const uint2*>(idx + o)) : make_uint2(0xffffffffu, 0xffffffffu);   // tap 255: nobody's
        g4[wy][wx] = live ? __ldg(reinterpret_cast<const uint4*>(dout + o)) : make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int py = 0; py < 2; ++py) {
      const int iy = 2 * a + py;
      if (iy >= H) continue;
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        const int ix = 2 * q + px;
        if (ix >= W) continue;
        float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        // an even row / column lies in one window row / column only (its centre), an odd one in two
#pragma unroll
        for (int wy = 0; wy <= py; ++wy) {
#pragma unroll
          for (int wx = 0; wx <= px; ++wx) {
            const uint32_t me = (uint32_t)((py + 1 - 2 * wy) * 3 + (px + 1 - 2 * wx));   // iy - (2*oy - 1), ix - (2*ox - 1)
            const uint32_t me4 = me * 0x01010101u;
            const uint32_t e0 = w8[wy][wx].x ^ me4, e1 = w8[wy][wx].y ^ me4;   // a zero byte = this window routes its gradient here
            float g[8];
            unpack_bf16x2(g4[wy][wx].x, g[0], g[1]); unpack_bf16x2(g4[wy][wx].y, g[2], g[3]);
            unpack_bf16x2(g4[wy][wx].z, g[4], g[5]); unpack_bf16x2(g4[wy][wx].w, g[6], g[7]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (((e0 >> (8 * j)) & 0xffu) == 0) acc[j] += g[j];
              if (((e1 >> (8 * j)) & 0xffu) == 0) acc[4 + j] += g[4 + j];
            }
          }
        }
        st8(dx + ((((long long)b * H + iy) * W + ix) * CG + cg) * 8, acc);
      }
    }
  }
}

// ---------------------------------------------------------------- zero insertion x2
__global__ void __launch_bounds__(256) zero_insert2x_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int B, int h,
                                                           int w, int C) {
  const int CG = C >> 3;
  const int H = 2 * h, W = 2 * w;
  const long long total = (long long)B * H * W * CG;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % CG);
    long long p = i / CG;
    const int X = (int)(p % W);
    p /= W;
    const int Y = (int)(p % H);
    const int b = (int)(p / H);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (((X | Y) & 1) == 0) v = __ldg(reinterpret_cast<const uint4*>(in + (((long long)b * h + (Y >> 1)) * w + (X >> 1)) * C + cg * 8));
    *reinterpret_cast<uint4*>(out + i * 8) = v;
  }
}

// ---------------------------------------------------------------- head backward
// dl[m, y, x] = sum_{Y,X} g[m, Y, X] * wy(Y, y) * wx(X, x), the transpose of ATen's align_corners bilinear
// (src = scale*dst, i0 = (int)src, i1 = i0 + (i0 < in-1), l1 = src - i0, l0 = 1 - l1).  One thread per low-res pixel.
__global__ void __launch_bounds__(128) upsample_bwd_kernel(const float* __restrict__ g, float* __restrict__ dl, int maps, int h, int w, int H,
                                                          int W, float ry, float rx) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= maps * h * w) return;
  const int x = idx % w, y = (idx / w) % h, m = idx / (w * h);
  // candidate source rows: ry*Y in (y-1, y+1)
  const float inv_ry = ry > 0.f ? 1.f / ry : 0.f, inv_rx = rx > 0.f ? 1.f / rx : 0.f;
  int Ylo = ry > 0.f ? max(0, (int)floorf((float)(y - 1) * inv_ry) - 1) : 0;
  int Yhi = ry > 0.f ? min(H - 1, (int)ceilf((float)(y + 1) * inv_ry) + 1) : H - 1;
  int Xlo = rx > 0.f ? max(0, (int)floorf((float)(x - 1) * inv_rx) - 1) : 0;
  int Xhi = rx > 0.f ? min(W - 1, (int)ceilf((float)(x + 1) * inv_rx) + 1) : W - 1;
  const float* gm = g + (size_t)m * H * W;
  float acc = 0.f;
  for (int Y = Ylo; Y <= Yhi; ++Y) {
    const float sy = ry * (float)Y;
    const int y0 = min((int)sy, h - 1);
    const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
    const float ly = sy - (float)y0, hy = 1.0f - ly;
    float wy = 0.f;
    if (y0 == y) wy += hy;
    if (y1 == y) wy += ly;
    if (wy == 0.f) continue;
    float rowacc = 0.f;
    for (int X = Xlo; X <= Xhi; ++X) {
      const float sx = rx * (float)X;
      const int x0 = min((int)sx, w - 1);
      const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
      const float lx = sx - (float)x0, hx = 1.0f - lx;
      float wx = 0.f;
      if (x0 == x) wx += hx;
      if (x1 == x) wx += lx;
      if (wx != 0.f) rowacc = fmaf(__ldg(gm + (size_t)Y * W + X), wx, rowacc);
    }
    acc = fmaf(rowacc, wy, acc);
  }
  dl[idx] = acc;
}

// The same transpose, separable and coalesced (round 2): one CTA per (map, low-res row y).  Phase 1: v[X] = sum_Y wy(Y, y) * g[m, Y, X] over the
// <= ~2*scale+3 high-res rows that touch y, every thread owning 4 consecutive X (float4 row reads); phase 2: dl[m, y, x] = sum_X wx(X, x) *
// v[X] from shared memory.  Each high-res row is read by the two CTAs whose low-res rows it feeds.  The one-thread-per-pixel kernel above
// spent ~4 k instructions per output on index arithmetic over 18 x 18 candidates with stride-8 loads: 190 us at batch 32 where this
// takes ~1/3 of that.  (Summation order: rows first, then columns.)
__global__ void __launch_bounds__(256) upsample_bwd_rows_kernel(const float* __restrict__ g, float* __restrict__ dl, int h, int w, int H, int W,
                                                               float ry, float rx) {
  extern __shared__ float v_row[];   // W floats (+ padding to a multiple of 4)
  const int y = blockIdx.x, m = blockIdx.y;
  const float inv_ry = ry > 0.f ? 1.f / ry : 0.f, inv_rx = rx > 0.f ? 1.f / rx : 0.f;
  const int Ylo = ry > 0.f ? max(0, (int)floorf((float)(y - 1) * inv_ry) - 1) : 0;
  const int Yhi = ry > 0.f ? min(H - 1, (int)ceilf((float)(y + 1) * inv_ry) + 1) : H - 1;
  const float* gm = g + (size_t)m * H * W;
  const bool vec = (W & 3) == 0;
  for (int X4 = threadIdx.x * 4; X4 < W; X4 += blockDim.x * 4) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int Y = Ylo; Y <= Yhi; ++Y) {
      const float sy = ry * (float)Y;
      const int y0 = min((int)sy, h - 1);
      const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
      const float ly = sy - (float)y0, hy = 1.0f - ly;
      float wy = 0.f;
      if (y0 == y) wy += hy;
      if (y1 == y) wy += ly;
      if (wy == 0.f) continue;   // CTA-uniform
      const float* row = gm + (size_t)Y * W + X4;
      if (vec) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(row));
        a0 = fmaf(q.x, wy, a0); a1 = fmaf(q.y, wy, a1); a2 = fmaf(q.z, wy, a2); a3 = fmaf(q.w, wy, a3);
      } else {
        a0 = fmaf(__ldg(row), wy, a0);
        if (X4 + 1 < W) a1 = fmaf(__ldg(row + 1), wy, a1);
        if (X4 + 2 < W) a2 = fmaf(__ldg(row + 2), wy, a2);
        if (X4 + 3 < W) a3 = fmaf(__ldg(row + 3), wy, a3);
      }
    }
    v_row[X4] = a0; v_row[X4 + 1] = a1; v_row[X4 + 2] = a2; v_row[X4 + 3] = a3;
  }
  __syncthreads();
  for (int x = threadIdx.x; x < w; x += blockDim.x) {
    const int Xlo = rx > 0.f ? max(0, (int)floorf((float)(x - 1) * inv_rx) - 1) : 0;
    const int Xhi = rx > 0.f ? min(W - 1, (int)ceilf((float)(x + 1) * inv_rx) + 1) : W - 1;
    float acc = 0.f;
    for (int X = Xlo; X <= Xhi; ++X) {
      const float sx = rx * (float)X;
      const int x0 = min((int)sx, w - 1);
      const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
      const float lx = sx - (float)x0, hx = 1.0f - lx;
      float wx = 0.f;
      if (x0 == x) wx += hx;
      if (x1 == x) wx += lx;
      if (wx != 0.f) acc = fmaf(v_row[X], wx, acc);
    }
    dl[((size_t)m * h + y) * w + x] = acc;
  }
}

// dfeat[p, c] = sum_k dl[b, k, pix] * w[k, c]   (bf16 NHWC out); one thread per (pixel, 8 channels)
__global__ void __launch_bounds__(256) fc_bwd_dfeat_kernel(const float* __restrict__ dl, const float* __restrict__ w_fc,
                                                          __nv_bfloat16* __restrict__ dfeat, int B, int K, int C, int hw) {
  const int CG = C >> 3;
  const long long total = (long long)B * hw * CG;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % CG);
    const long long p = i / CG;
    const int b = (int)(p / hw), pix = (int)(p - (long long)b * hw);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int k = 0; k < K; ++k) {
      const float d = __ldg(dl + ((size_t)b * K + k) * hw + pix);
      const float4 a = __ldg(reinterpret_cast<const float4*>(w_fc + (size_t)k * C + cg * 8));
      const float4 c = __ldg(reinterpret_cast<const float4*>(w_fc + (size_t)k * C + cg * 8 + 4));
      acc[0] = fmaf(d, a.x, acc[0]); acc[1] = fmaf(d, a.y, acc[1]); acc[2] = fmaf(d, a.z, acc[2]); acc[3] = fmaf(d, a.w, acc[3]);
      acc[4] = fmaf(d, c.x, acc[4]); acc[5] = fmaf(d, c.y, acc[5]); acc[6] = fmaf(d, c.z, acc[6]); acc[7] = fmaf(d, c.w, acc[7]);
    }
    st8(dfeat + i * 8, acc);
  }
}

// partial[blk][k][c] = sum over the block's pixel slab of dl[b,k,pix] * feat[p,c];  thread = one channel pair, 4 keypoints at a time
constexpr int FCW_SLAB = 64;
__global__ void __launch_bounds__(256) fc_bwd_dw_partial_kernel(const float* __restrict__ dl, const __nv_bfloat16* __restrict__ feat,
                                                               float* __restrict__ partial, int B, int K, int C, int hw) {
  __shared__ float sdl[4][FCW_SLAB];
  const long long P = (long long)B * hw;
  const long long p0 = (long long)blockIdx.x * FCW_SLAB;
  const int n = (int)min((long long)FCW_SLAB, P - p0);
  for (int kg = 0; kg < K; kg += 4) {
    __syncthreads();
    for (int t = threadIdx.x; t < 4 * FCW_SLAB; t += blockDim.x) {
      const int j = t / FCW_SLAB, q = t - j * FCW_SLAB;
      float v = 0.f;
      if (q < n && kg + j < K) {
        const long long p = p0 + q;
        const int b = (int)(p / hw), pix = (int)(p - (long long)b * hw);
        v = dl[((size_t)b * K + kg + j) * hw + pix];
      }
      sdl[j][q] = v;
    }
    __syncthreads();
    for (int c = threadIdx.x * 2; c < C; c += blockDim.x * 2) {
      float acc[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
      for (int q = 0; q < n; ++q) {
        float f0, f1;
        unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(feat + (p0 + q) * C + c)), f0, f1);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[j][0] = fmaf(sdl[j][q], f0, acc[j][0]);
          acc[j][1] = fmaf(sdl[j][q], f1, acc[j][1]);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (kg + j < K) {
          partial[((size_t)blockIdx.x * K + kg + j) * C + c] = acc[j][0];
          partial[((size_t)blockIdx.x * K + kg + j) * C + c + 1] = acc[j][1];
        }
    }
  }
}
// dw[k][c] = sum_blk partial   (grid: (C/32, K); 256 threads = 32 channels x 8 slices of the blocks)
__global__ void __launch_bounds__(256) fc_bwd_dw_finalize_kernel(const float* __restrict__ partial, int nblk, float* __restrict__ dw, int K, int C,
                                                                int accumulate) {
  __shared__ double sh[8][32];
  const int k = blockIdx.y, c = blockIdx.x * 32 + (threadIdx.x & 31), slice = threadIdx.x >> 5;
  float a0 = 0.f, a1 = 0.f;
  int b = slice;
  for (; b + 8 < nblk; b += 16) {
    a0 += partial[((size_t)b * K + k) * C + c];
    a1 += partial[((size_t)(b + 8) * K + k) * C + c];
  }
  if (b < nblk) a0 += partial[((size_t)b * K + k) * C + c];
  sh[slice][threadIdx.x & 31] = (double)a0 + (double)a1;
  __syncthreads();
  if (threadIdx.x < 32) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += sh[i][threadIdx.x];
    dw[(size_t)k * C + c] = (accumulate ? dw[(size_t)k * C + c] : 0.f) + (float)s;
  }
}
// db[k] = sum_{b,pix} dl[b,k,pix] in two fixed-order stages: one block per (k, b) map, then one thread per k over the B partials
// (a single block per k walking all B*hw elements serially cost 0.29 ms at B = 32)
__global__ void __launch_bounds__(256) fc_bwd_db_partial_kernel(const float* __restrict__ dl, double* __restrict__ partial, int K, int hw) {
  const int k = blockIdx.x, b = blockIdx.y;
  const float* src = dl + ((size_t)b * K + k) * hw;
  __shared__ double red[256];
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int i = threadIdx.x;
  for (; i + 3 * 256 < hw; i += 4 * 256) {
    s0 += src[i]; s1 += src[i + 256]; s2 += src[i + 512]; s3 += src[i + 768];
  }
  for (; i < hw; i += 256) s0 += src[i];
  red[threadIdx.x] = ((double)s0 + (double)s1) + ((double)s2 + (double)s3);
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (threadIdx.x < st) red[threadIdx.x] += red[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[(size_t)b * K + k] = red[0];
}
__global__ void fc_bwd_db_final_kernel(const double* __restrict__ partial, float* __restrict__ db, int B, int K, int accumulate) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  double s = 0.0;
  for (int b = 0; b < B; ++b) s += partial[(size_t)b * K + k];
  db[k] = (accumulate ? db[k] : 0.f) + (float)s;
}

static int grid_for(long long n, int threads) {
  long long blocks = ceil_div_ll(n, threads);
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace hk

extern "C" {

int hk_maxpool3x3s2_bwd(const void* dout, const void* x, void* dx, int B, int H, int W, int C, int Ho, int Wo, void* idx_ws,
                        size_t idx_ws_bytes, void* stream) {
  using namespace hk;
  HK_REQUIRE(dout && x && dx && idx_ws, "hk_maxpool3x3s2_bwd: null pointer");
  HK_REQUIRE(idx_ws_bytes >= (size_t)B * Ho * Wo * C, "hk_maxpool3x3s2_bwd: index workspace too small (B*Ho*Wo*C bytes)");
  HK_REQUIRE(B > 0 && H > 0 && W > 0 && C >= 8 && (C & 7) == 0 && Ho == (H + 2 - 3) / 2 + 1 && Wo == (W + 2 - 3) / 2 + 1,
             "hk_maxpool3x3s2_bwd: bad shape");
  maxpool_argmax_kernel<<<grid_for((long long)B * Ho * Wo * (C >> 3), 256), 256, 0, as_stream(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<uint8_t*>(idx_ws), B, H, W, C, Ho, Wo);
  int rc = check_launch("maxpool_argmax_kernel");
  if (rc) return rc;
  const long long total = (long long)B * ((H + 1) / 2) * ((W + 1) / 2) * (C >> 3);
  maxpool_bwd_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(static_cast<const __nv_bfloat16*>(dout),
                                                                         static_cast<const uint8_t*>(idx_ws),
                                                                         static_cast<__nv_bfloat16*>(dx), B, H, W, C, Ho, Wo);
  return check_launch("maxpool_bwd_kernel");
}

// Training-step max-pool in two halves: the forward also records which tap of every window won (ATen's max_pool2d_with_indices rule: first
// maximum in scan order), the backward is then the gather alone.
int hk_maxpool3x3s2_fwd_idx(const void* x, void* y, void* idx, int B, int H, int W, int C, int Ho, int Wo, void* stream) {
  using namespace hk;
  HK_REQUIRE(x && y && idx, "hk_maxpool3x3s2_fwd_idx: null pointer");
  HK_REQUIRE(B > 0 && H > 0 && W > 0 && C >= 8 && (C & 7) == 0 && Ho == (H + 2 - 3) / 2 + 1 && Wo == (W + 2 - 3) / 2 + 1,
             "hk_maxpool3x3s2_fwd_idx: bad shape");
  maxpool_argmax_kernel<<<grid_for((long long)B * Ho * Wo * (C >> 3), 256), 256, 0, as_stream(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<uint8_t*>(idx), B, H, W, C, Ho, Wo, static_cast<__nv_bfloat16*>(y));
  return check_launch("maxpool_argmax_kernel");
}

int hk_maxpool3x3s2_bwd_idx(const void* dout, const void* idx, void* dx, int B, int H, int W, int C, int Ho, int Wo, void* stream) {
  using namespace hk;
  HK_REQUIRE(dout && idx && dx, "hk_maxpool3x3s2_bwd_idx: null pointer");
  HK_REQUIRE(B > 0 && H > 0 && W > 0 && C >= 8 && (C & 7) == 0 && Ho == (H + 2 - 3) / 2 + 1 && Wo == (W + 2 - 3) / 2 + 1,
             "hk_maxpool3x3s2_bwd_idx: bad shape");
  const long long total = (long long)B * ((H + 1) / 2) * ((W + 1) / 2) * (C >> 3);
  maxpool_bwd_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(static_cast<const __nv_bfloat16*>(dout), static_cast<const uint8_t*>(idx),
                                                                         static_cast<__nv_bfloat16*>(dx), B, H, W, C, Ho, Wo);
  return check_launch("maxpool_bwd_kernel");
}

int hk_zero_insert2x(const void* in, void* out, int B, int h, int w, int C, void* stream) {
  using namespace hk;
  HK_REQUIRE(in && out && B > 0 && h > 0 && w > 0 && C >= 8 && (C & 7) == 0, "hk_zero_insert2x: bad argument");
  const long long total = (long long)B * 2 * h * 2 * w * (C >> 3);
  zero_insert2x_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(static_cast<const __nv_bfloat16*>(in),
                                                                           static_cast<__nv_bfloat16*>(out), B, h, w, C);
  return check_launch("zero_insert2x_kernel");
}

size_t hk_head_bwd_workspace_bytes(int B, int K, int C, int h, int w) {
  const long long P = (long long)B * h * w;
  const long long nblk = (P + hk::FCW_SLAB - 1) / hk::FCW_SLAB;
  return (size_t)nblk * K * C * sizeof(float);
}

int hk_head_bwd(const float* g_up, const void* feat, const float* w_fc, float* dlogits_ws, void* dfeat, float* dw_fc, float* db_fc,
                int accumulate, int B, int K, int C, int h, int w, int H, int W, void* ws, size_t ws_bytes, void* stream) {
  using namespace hk;
  HK_REQUIRE(g_up && feat && w_fc && dlogits_ws && ws, "hk_head_bwd: null pointer");
  HK_REQUIRE(B > 0 && K > 0 && C >= 8 && (C & 7) == 0 && h > 0 && w > 0 && H > 0 && W > 0, "hk_head_bwd: bad shape");
  HK_REQUIRE(ws_bytes >= hk_head_bwd_workspace_bytes(B, K, C, h, w), "hk_head_bwd: workspace too small");
  HK_REQUIRE((long long)B * K * h * w < 0x7fffffffLL, "hk_head_bwd: too many low-res elements");
  cudaStream_t s = as_stream(stream);
  const float ry = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f;
  const float rx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
  const int n = B * K * h * w;
  int rc;
  const size_t vbytes = (size_t)((W + 3) / 4 * 4) * sizeof(float);
  if (h <= 65535 && B * K <= 65535 && vbytes <= 48 * 1024 && (reinterpret_cast<uintptr_t>(g_up) & 15) == 0) {
    upsample_bwd_rows_kernel<<<dim3(h, B * K), 256, vbytes, s>>>(g_up, dlogits_ws, h, w, H, W, ry, rx);
    rc = check_launch("upsample_bwd_rows_kernel");
  } else {
    upsample_bwd_kernel<<<ceil_div(n, 128), 128, 0, s>>>(g_up, dlogits_ws, B * K, h, w, H, W, ry, rx);
    rc = check_launch("upsample_bwd_kernel");
  }
  if (rc) return rc;
  const int hw = h * w;
  if (dfeat) {
    fc_bwd_dfeat_kernel<<<grid_for((long long)B * hw * (C >> 3), 256), 256, 0, s>>>(dlogits_ws, w_fc, static_cast<__nv_bfloat16*>(dfeat), B,
                                                                                   K, C, hw);
    rc = check_launch("fc_bwd_dfeat_kernel");
    if (rc) return rc;
  }
  if (dw_fc) {
    const int nblk = (int)(((long long)B * hw + FCW_SLAB - 1) / FCW_SLAB);
    fc_bwd_dw_partial_kernel<<<nblk, 256, 0, s>>>(dlogits_ws, static_cast<const __nv_bfloat16*>(feat), static_cast<float*>(ws), B, K, C, hw);
    rc = check_launch("fc_bwd_dw_partial_kernel");
    if (rc) return rc;
    HK_REQUIRE(C % 32 == 0, "hk_head_bwd: C must be a multiple of 32");
    fc_bwd_dw_finalize_kernel<<<dim3(C / 32, K), 256, 0, s>>>(static_cast<const float*>(ws), nblk, dw_fc, K, C, accumulate);
    rc = check_launch("fc_bwd_dw_finalize_kernel");
    if (rc) return rc;
  }
  if (!db_fc) return 0;
  // the dw partials in `ws` are consumed: its head is reused for the B x K double partials of db
  HK_REQUIRE(ws_bytes >= (size_t)B * K * sizeof(double) && (reinterpret_cast<uintptr_t>(ws) & 7) == 0, "hk_head_bwd: workspace too small for db");
  fc_bwd_db_partial_kernel<<<dim3(K, B), 256, 0, s>>>(dlogits_ws, static_cast<double*>(ws), K, hw);
  rc = check_launch("fc_bwd_db_partial_kernel");
  if (rc) return rc;
  fc_bwd_db_final_kernel<<<ceil_div(K, 64), 64, 0, s>>>(static_cast<const double*>(ws), db_fc, B, K, accumulate);
  return check_launch("fc_bwd_db_final_kernel");
}

}  // extern "C"
