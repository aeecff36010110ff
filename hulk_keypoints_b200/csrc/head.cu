// Heatmap head (SURVEY.md k8 + k9): scoring 1x1 conv on the K live rows, bilinear x8 upsample with
// align_corners=True, sigmoid.  HBM-bound: reads the (B,h,w,C) feature map once, writes (B,K,H,W) fp32 once.
//
// Reference call sites: src/resnet.py:215 (fc applied as a 1x1 conv), src/resnet_dilated.py:27
// (upsample_bilinear to the input size), src/model.py:21 (slice [:, :K], sigmoid).  The reference runs
// the conv and the upsample on all 1000 channels and slices afterwards; both ops act per output
// channel, so only the K kept rows are computed here.
//
//   1. head_logits_kernel: one warp per low-res pixel (two pixels in flight per warp); 128-bit loads of the
//      C-vector; fc rows live in REGISTERS in groups of 4 keypoints (the config.py case K=4 needs one
//      group); a 6-shuffle multi-value butterfly reduces the 4 dot products -> (B,K,h,w) fp32 logits, which
//      stay L2-resident for step 2.
//   2. head_upsample_sigmoid_kernel: one thread per 4 consecutive output x; ATen's align_corners
//      arithmetic (scale=(in-1)/(out-1), src=scale*dst, lambda=src-floor) in fp32, sigmoid, float4 store.
//      All index math is 32-bit (64-bit div/mod was the bottleneck of the first version).
#include "hk_common.cuh"

namespace hk {

constexpr int kHeadThreads = 256;
constexpr int kHeadMaxPerLane = 16;  // C <= 512

// 8 consecutive channels held RAW in registers (bf16: one uint4; fp32: two float4) and unpacked at first use, so
// several pixels' loads can be in flight without doubling the register footprint.
template <typename FeatT>
struct Raw8;
template <>
struct Raw8<__nv_bfloat16> {
  uint4 q;
  __device__ __forceinline__ void load(const __nv_bfloat16* p) { q = __ldcs(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ void unpack(float* f) const {
    unpack_bf16x2(q.x, f[0], f[1]);
    unpack_bf16x2(q.y, f[2], f[3]);
    unpack_bf16x2(q.z, f[4], f[5]);
    unpack_bf16x2(q.w, f[6], f[7]);
  }
};
template <>
struct Raw8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p) {
    a = __ldcs(reinterpret_cast<const float4*>(p));
    b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
  }
  __device__ __forceinline__ void unpack(float* f) const {
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
    f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
};

// Sum v[0..3] over the 32 lanes with 6 shuffles; afterwards lane 8*k holds the total of v[k].
__device__ __forceinline__ float reduce4(const float (&v)[4], int lane) {
  const bool hi = (lane & 16) != 0;
  float k0 = hi ? v[2] : v[0], k1 = hi ? v[3] : v[1];
  const float s0 = hi ? v[0] : v[2], s1 = hi ? v[1] : v[3];
  k0 += __shfl_xor_sync(0xffffffffu, s0, 16);
  k1 += __shfl_xor_sync(0xffffffffu, s1, 16);
  const bool hi2 = (lane & 8) != 0;
  float kk = hi2 ? k1 : k0;
  const float s = hi2 ? k0 : k1;
  kk += __shfl_xor_sync(0xffffffffu, s, 8);
  kk += __shfl_xor_sync(0xffffffffu, kk, 4);
  kk += __shfl_xor_sync(0xffffffffu, kk, 2);
  kk += __shfl_xor_sync(0xffffffffu, kk, 1);
  return kk;
}

// SLABS = C / 256 (1 or 2).  Keypoints are processed in groups of 4 (weights of the group in registers).
template <typename FeatT, int SLABS>
__global__ void __launch_bounds__(kHeadThreads)
head_logits_kernel(const FeatT* __restrict__ feat, const float* __restrict__ w_fc, const float* __restrict__ b_fc,
                   float* __restrict__ logits, int pixels, int hw, int K, int C) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = kHeadThreads >> 5;
  const int wstride = gridDim.x * warps_per_block;
  constexpr int PER = SLABS * 8;
  for (int kg = 0; kg < K; kg += 4) {
    float wr[4][PER];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = min(kg + j, K - 1);
#pragma unroll
      for (int s = 0; s < SLABS; ++s) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(w_fc + (size_t)k * C + s * 256 + lane * 8));
        const float4 b = __ldg(reinterpret_cast<const float4*>(w_fc + (size_t)k * C + s * 256 + lane * 8 + 4));
        wr[j][s * 8 + 0] = a.x; wr[j][s * 8 + 1] = a.y; wr[j][s * 8 + 2] = a.z; wr[j][s * 8 + 3] = a.w;
        wr[j][s * 8 + 4] = b.x; wr[j][s * 8 + 5] = b.y; wr[j][s * 8 + 6] = b.z; wr[j][s * 8 + 7] = b.w;
      }
    }
    const int kq = kg + (lane >> 3);  // keypoint whose total lands in this lane (lanes 0, 8, 16, 24)
    const float bq = (kq < K) ? __ldg(b_fc + kq) : 0.f;
    // NPIX pixels in flight per warp: all feature loads are issued before the first use (HBM latency hiding)
    constexpr int NPIX = sizeof(FeatT) == 2 ? 4 : 2;
    for (int pix0 = blockIdx.x * warps_per_block + (threadIdx.x >> 5); pix0 < pixels; pix0 += NPIX * wstride) {
      Raw8<FeatT> raw[NPIX][SLABS];
#pragma unroll
      for (int p = 0; p < NPIX; ++p) {
        const int pix = pix0 + p * wstride;
        if (pix < pixels) {
#pragma unroll
          for (int s = 0; s < SLABS; ++s) raw[p][s].load(feat + (size_t)pix * C + s * 256 + lane * 8);
        }
      }
#pragma unroll
      for (int p = 0; p < NPIX; ++p) {
        const int pix = pix0 + p * wstride;
        if (pix < pixels) {  // warp-uniform
          float f[PER];
#pragma unroll
          for (int s = 0; s < SLABS; ++s) raw[p][s].unpack(f + s * 8);
          float acc[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc[j] = 0.f;
#pragma unroll
            for (int i = 0; i < PER; ++i) acc[j] = fmaf(f[i], wr[j][i], acc[j]);
          }
          const float r = reduce4(acc, lane);
          if ((lane & 7) == 0 && kq < K) {
            const int b = pix / hw, rem = pix - b * hw;
            logits[((size_t)b * K + kq) * hw + rem] = r + bq;
          }
        }
      }
    }
  }
}

template <bool FAST>
__device__ __forceinline__ float sigmoid_f(float v) {
  if (FAST) return __fdividef(1.0f, 1.0f + __expf(-v));
  return 1.0f / (1.0f + expf(-v));
}

// One CTA = one output row (map = blockIdx.z, Y = blockIdx.y); one thread = 4 consecutive output x.  The two source
// rows are staged in shared memory; no integer division anywhere.  FAST (bf16 mode): the vertical lerp is done once
// per source column while staging (separable form); exact (fp32 mode): ATen's operation order
// hy*(hx*a + lx*b) + ly*(hx*c + lx*d) is kept so the result tracks the reference to the last ulp or two.
template <bool FAST, bool SIGMOID = true>
__global__ void __launch_bounds__(256)
head_upsample_sigmoid_kernel(const float* __restrict__ logits, float* __restrict__ heat, int h, int w, int H, int W,
                             int wq, float ry, float rx) {
  extern __shared__ float srow[];  // FAST: w floats; exact: 2*w floats
  const int map = blockIdx.z, Y = blockIdx.y;
  const float sy = ry * (float)Y;
  const int y0 = min((int)sy, h - 1);
  const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
  const float ly = sy - (float)y0, hy = 1.0f - ly;
  const float* row0 = logits + ((size_t)map * h + y0) * w;
  const float* row1 = logits + ((size_t)map * h + y1) * w;
  for (int i = threadIdx.x; i < w; i += blockDim.x) {
    const float a = __ldg(row0 + i), c = __ldg(row1 + i);
    if (FAST) {
      srow[i] = hy * a + ly * c;
    } else {
      srow[i] = a;
      srow[w + i] = c;
    }
  }
  __syncthreads();
  const int xq = blockIdx.x * blockDim.x + threadIdx.x;
  if (xq >= wq) return;
  float o[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int X = min(xq * 4 + j, W - 1);
    const float sx = rx * (float)X;
    const int x0 = min((int)sx, w - 1);
    const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
    const float lx = sx - (float)x0, hx = 1.0f - lx;
    float v;
    if (FAST) v = hx * srow[x0] + lx * srow[x1];
    else v = hy * (hx * srow[x0] + lx * srow[x1]) + ly * (hx * srow[w + x0] + lx * srow[w + x1]);
    o[j] = SIGMOID ? sigmoid_f<FAST>(v) : v;
  }
  float* dst = heat + ((size_t)map * H + Y) * W + xq * 4;
  if ((W & 3) == 0) {
    __stcs(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (xq * 4 + j < W) dst[j] = o[j];
  }
}

// ---- throughput-mode upsample: ROWS output rows per CTA, the x interpolation set-up amortised over them, optional fused argmax ----
constexpr int kHeadRows = 32;   // rows-per-CTA sweep at 480x640 (B200): 8: 0.084 ms, 16: 0.077, 32: 0.076, 60: 0.078
// grid (ceil(H / kHeadRows), B*K); each thread owns 4 consecutive output x (loops when W/4 > blockDim).  The source rows touched by the
// CTA's output rows are staged once; per row three vertical lerps (the 4 outputs of a thread read at most 3 consecutive source columns)
// and one horizontal lerp + sigmoid per output (the separable form of the kernel above).  (Fusing the argmax into this kernel was
// measured and dropped: the kernel is instruction-bound and the compare cost more than the stand-alone decode's HBM read.)
__global__ void __launch_bounds__(256)
head_upsample_rows_kernel(const float* __restrict__ logits, float* __restrict__ heat, int h, int w, int H, int W, int wq, float ry, float rx,
                          int nsrc, int rows_per_cta) {
  extern __shared__ float srows[];  // nsrc x w
  const int map = blockIdx.y;
  const int Y0 = blockIdx.x * rows_per_cta;
  const int Yend = min(H, Y0 + rows_per_cta);
  const int ybase = min((int)(ry * (float)Y0), h - 1);
  const float* src = logits + (size_t)map * h * w;
  for (int i = threadIdx.x; i < nsrc * w; i += blockDim.x) {
    const int r = i / w, c = i - r * w;
    srows[i] = __ldg(src + (size_t)min(ybase + r, h - 1) * w + c);
  }
  __syncthreads();
  for (int xq = threadIdx.x; xq < wq; xq += blockDim.x) {
    // x set-up once per thread, reused by all rows: the 4 outputs read at most 3 consecutive source columns c0, c0+1, c0+2
    float lx[4], hx[4];
    bool a1[4], b1[4], b2[4];   // left tap = column c0 + a1; right tap = column c0 + b1 + b2  (b2 implies b1)
    int c0 = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int X = min(xq * 4 + j, W - 1);
      const float sx = rx * (float)X;
      const int x0 = min((int)sx, w - 1);
      const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
      if (j == 0) c0 = x0;
      lx[j] = sx - (float)x0;
      hx[j] = 1.0f - lx[j];
      a1[j] = x0 - c0 >= 1;        // x0 - c0 in {0, 1}: 3*rx < 1 is checked on the host
      b1[j] = x1 - c0 >= 1;        // x1 - c0 in {0, 1, 2}
      b2[j] = x1 - c0 >= 2;
    }
    const int c1 = min(c0 + 1, w - 1), c2 = min(c0 + 2, w - 1);
    for (int Y = Y0; Y < Yend; ++Y) {
      const float sy = ry * (float)Y;
      const int y0 = min((int)sy, h - 1);
      const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
      const float ly = sy - (float)y0, hy = 1.0f - ly;
      const float* r0 = srows + (y0 - ybase) * w;
      const float* r1 = srows + (y1 - ybase) * w;
      const float t0 = hy * r0[c0] + ly * r1[c0];
      const float t1 = hy * r0[c1] + ly * r1[c1];
      const float t2 = hy * r0[c2] + ly * r1[c2];
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float ta = a1[j] ? t1 : t0;
        const float tb = b2[j] ? t2 : (b1[j] ? t1 : t0);
        o[j] = sigmoid_f<true>(hx[j] * ta + lx[j] * tb);
      }
      float* dst = heat + ((size_t)map * H + Y) * W + xq * 4;
      if ((W & 3) == 0) {
        __stcs(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (xq * 4 + j < W) dst[j] = o[j];
      }
    }
  }
}

template <typename FeatT>
static void launch_logits(const void* feat, const float* w_fc, const float* b_fc, float* logits, int pixels, int hw, int K, int C,
                          cudaStream_t s) {
  int blocks = ceil_div(pixels, (kHeadThreads / 32) * 4);
  const int cap = sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (C == 512)
    head_logits_kernel<FeatT, 2><<<blocks, kHeadThreads, 0, s>>>(static_cast<const FeatT*>(feat), w_fc, b_fc, logits, pixels, hw, K, C);
  else
    head_logits_kernel<FeatT, 1><<<blocks, kHeadThreads, 0, s>>>(static_cast<const FeatT*>(feat), w_fc, b_fc, logits, pixels, hw, K, C);
}

}  // namespace hk

static int head_fwd_impl(const void* feat, int feat_dtype, const float* w_fc, const float* b_fc, float* logits_ws, float* heat, int B,
                         int K, int C, int h, int w, int H, int W, bool sigmoid, void* stream);
static int head_upsample_impl(const float* logits_ws, float* heat, int B, int K, int h, int w, int H, int W, bool sigmoid, bool fast, void* stream);

// x8 bilinear upsample (align_corners=True) + sigmoid of (B,K,h,w) fp32 logits that are already there -- the second half of hk_head_fwd,
// for logits produced by hk_conv_head_fwd.  fast != 0: the throughput-mode arithmetic of the bf16 path; 0: ATen's exact operation order.
extern "C" int hk_head_upsample_fwd(const float* logits, float* heat, int B, int K, int h, int w, int H, int W, int fast, void* stream) {
  using namespace hk;
  HK_REQUIRE(logits && heat, "hk_head_upsample_fwd: null pointer");
  HK_REQUIRE(B > 0 && K > 0 && h > 0 && w > 0 && H > 0 && W > 0, "hk_head_upsample_fwd: bad shape");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(heat) & 15) == 0, "hk_head_upsample_fwd: heat must be 16-byte aligned");
  return head_upsample_impl(logits, heat, B, K, h, w, H, W, true, fast != 0, stream);
}

extern "C" int hk_head_fwd(const void* feat, int feat_dtype, const float* w_fc, const float* b_fc, float* logits_ws,
                           float* heat, int B, int K, int C, int h, int w, int H, int W, void* stream) {
  return head_fwd_impl(feat, feat_dtype, w_fc, b_fc, logits_ws, heat, B, K, C, h, w, H, W, true, stream);
}

extern "C" int hk_head_logits_fwd(const void* feat, int feat_dtype, const float* w_fc, const float* b_fc, float* logits_ws,
                                  float* logits_up, int B, int K, int C, int h, int w, int H, int W, void* stream) {
  return head_fwd_impl(feat, feat_dtype, w_fc, b_fc, logits_ws, logits_up, B, K, C, h, w, H, W, false, stream);
}

static int head_fwd_impl(const void* feat, int feat_dtype, const float* w_fc, const float* b_fc, float* logits_ws, float* heat, int B,
                         int K, int C, int h, int w, int H, int W, bool sigmoid, void* stream) {
  using namespace hk;
  HK_REQUIRE(feat && w_fc && b_fc && logits_ws && heat, "hk_head_fwd: null pointer");
  HK_REQUIRE(B > 0 && K > 0 && h > 0 && w > 0 && H > 0 && W > 0, "hk_head_fwd: bad shape");
  HK_REQUIRE(C == 256 || C == 512, "hk_head_fwd: C=%d must be 256 or 512", C);
  HK_REQUIRE(feat_dtype == HK_BF16 || feat_dtype == HK_F32, "hk_head_fwd: feat dtype must be bf16 or f32");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(feat) & 15) == 0 && (reinterpret_cast<uintptr_t>(heat) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(w_fc) & 15) == 0,
             "hk_head_fwd: feat/heat/w_fc must be 16-byte aligned");
  HK_REQUIRE((long long)B * h * w < 0x7fffffffLL, "hk_head_fwd: too many low-res pixels");
  cudaStream_t s = as_stream(stream);
  const int pixels = B * h * w;
  if (feat_dtype == HK_BF16) launch_logits<__nv_bfloat16>(feat, w_fc, b_fc, logits_ws, pixels, h * w, K, C, s);
  else launch_logits<float>(feat, w_fc, b_fc, logits_ws, pixels, h * w, K, C, s);
  int rc = check_launch("head_logits_kernel");
  if (rc) return rc;
  return head_upsample_impl(logits_ws, heat, B, K, h, w, H, W, sigmoid, feat_dtype == HK_BF16, stream);
}

static int head_upsample_impl(const float* logits_ws, float* heat, int B, int K, int h, int w, int H, int W, bool sigmoid, bool fast, void* stream) {
  using namespace hk;
  cudaStream_t s = as_stream(stream);
  // ATen area_pixel_compute_scale(align_corners=True): (in - 1) / (out - 1) in float, 0 when out == 1
  const float ry = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f;
  const float rx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
  const int wq = (W + 3) / 4;
  HK_REQUIRE(H <= 65535 && B * K <= 65535 && w <= 4096, "hk_head_fwd: H, B*K or w exceed the launch grid limits");
  int threads = ((wq + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  dim3 grid(ceil_div(wq, threads), H, B * K);
  // bf16 features = throughput mode: separable lerp + ex2/rcp-approx sigmoid; fp32 features = correctness mode
  if (!sigmoid)  // training: upsampled logits in ATen's exact operation order; the sigmoid lives in hk_bce_fwd_bwd
    head_upsample_sigmoid_kernel<false, false><<<grid, threads, (size_t)2 * w * sizeof(float), s>>>(logits_ws, heat, h, w, H, W, wq, ry, rx);
  else if (fast && 3.0f * rx < 1.0f) {   // (the rows kernel assumes <= 3 source columns per 4 outputs)
    const int nsrc = (int)(ry * (float)kHeadRows) + 3;
    const dim3 grid2(ceil_div(H, kHeadRows), B * K);
    const size_t smem = (size_t)nsrc * w * sizeof(float);
    HK_REQUIRE(smem <= 48 * 1024, "hk_head_fwd: low-res row too wide for the staging buffer");
    head_upsample_rows_kernel<<<grid2, threads, smem, s>>>(logits_ws, heat, h, w, H, W, wq, ry, rx, nsrc, kHeadRows);
    return check_launch("head_upsample_rows_kernel");
  } else if (fast)
    head_upsample_sigmoid_kernel<true><<<grid, threads, (size_t)w * sizeof(float), s>>>(logits_ws, heat, h, w, H, W, wq, ry, rx);
  else
    head_upsample_sigmoid_kernel<false><<<grid, threads, (size_t)2 * w * sizeof(float), s>>>(logits_ws, heat, h, w, H, W, wq, ry, rx);
  return check_launch("head_upsample_sigmoid_kernel");
}
