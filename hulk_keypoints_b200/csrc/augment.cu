// Training-batch augmentation on the device: a random affine warp of each image with its keypoint labels moved by the same map, and
// photometric jitter (contrast, brightness, per-channel gain, Gaussian noise).  Replaces the reference's domain-randomisation pipeline
// (src/dataset.py:18-31, imgaug, commented out there) and, for warped labels, the clipping of :63-66.
//
// The host (hulk_keypoints_b200/augment.py) draws per image `tries` candidate geometries as 2x3 matrices, forward (label map) and inverse
// (image sampling map), computed in fp64 and rounded once to fp32; these kernels only read them.
//   hk_augment_pick   : per image the first candidate that keeps all K labels inside [0, W-1] x [0, H-1] (-1: none, identity geometry)
//                       and the moved labels.  One thread per image.
//   hk_augment_images : out(p) = bilinear(in, Ainv(p)) (grid_sample, align_corners=True, zero padding), then per channel
//                       v = (v - 0.5)*c + 0.5 + beta;  v *= g_ch;  v += noise_std*n;  v = clamp(v, 0, 1).
//                       Bound: HBM (12 B read + 12 B written per pixel, plus gather overfetch under rotation).
#include "hk_common.cuh"

namespace hk {

constexpr int kAugThreads = 256;

// Random123's Philox4x32-10 (Salmon et al., SC'11): counter c, key (k0, k1), ten rounds.
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c[0], hi0 = __umulhi(0xD2511F53u, c[0]);
    const uint32_t lo1 = 0xCD9E8D57u * c[2], hi1 = __umulhi(0xCD9E8D57u, c[2]);
    c[0] = hi1 ^ c[1] ^ k0;
    c[1] = lo1;
    c[2] = hi0 ^ c[3] ^ k1;
    c[3] = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}

// 23 random bits -> (m + 0.5) * 2^-23: exact in fp32, strictly inside (0, 1), so the logarithm below is finite.
__device__ __forceinline__ float uniform_open(uint32_t r) { return ((float)(r >> 9) + 0.5f) * 0x1p-23f; }

// One Philox output -> four N(0,1) values (two Box-Muller pairs).  logf / sqrtf / sincospif, not the fast intrinsics, so that a float64
// restatement of the same formula agrees to ~1e-6.
__device__ __forceinline__ void normals4(uint32_t xq, uint32_t y, uint32_t ch, uint32_t b, uint32_t k0, uint32_t k1, float n[4]) {
  uint32_t c[4] = {xq, y, ch, b};
  philox4x32_10(c, k0, k1);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float rad = sqrtf(-2.0f * logf(uniform_open(c[2 * i])));
    float s, co;
    sincospif(2.0f * uniform_open(c[2 * i + 1]), &s, &co);
    n[2 * i] = rad * co;
    n[2 * i + 1] = rad * s;
  }
}

// m (2x3 row-major) applied to (x, y) with one fp32 rounding per operation, in this order: (m0*x + m1*y) + m2.  The test restatement
// repeats the same sequence in numpy fp32, so the in-frame decision agrees bit for bit.
__device__ __forceinline__ float affine_rn(float m0, float m1, float m2, float x, float y) {
  return __fadd_rn(__fadd_rn(__fmul_rn(m0, x), __fmul_rn(m1, y)), m2);
}

__global__ void augment_pick_kernel(const float* __restrict__ fwd, int B, int tries, int K, float xmax, float ymax,
                                    const float* __restrict__ uv, float* __restrict__ uv_out, int32_t* __restrict__ pick) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* u = uv + (size_t)b * K * 2;
  int chosen = -1;
  for (int t = 0; t < tries && chosen < 0; ++t) {
    const float* m = fwd + ((size_t)b * tries + t) * 6;
    bool ok = true;
    for (int k = 0; k < K && ok; ++k) {
      const float x = u[2 * k], y = u[2 * k + 1];
      const float xp = affine_rn(m[0], m[1], m[2], x, y), yp = affine_rn(m[3], m[4], m[5], x, y);
      ok = xp >= 0.f && xp <= xmax && yp >= 0.f && yp <= ymax;   // false for NaN
    }
    if (ok) chosen = t;
  }
  pick[b] = chosen;
  float* o = uv_out + (size_t)b * K * 2;
  if (chosen < 0) {
    for (int k = 0; k < 2 * K; ++k) o[k] = u[k];
    return;
  }
  const float* m = fwd + ((size_t)b * tries + chosen) * 6;
  for (int k = 0; k < K; ++k) {
    const float x = u[2 * k], y = u[2 * k + 1];
    o[2 * k] = affine_rn(m[0], m[1], m[2], x, y);
    o[2 * k + 1] = affine_rn(m[3], m[4], m[5], x, y);
  }
}

// grid (ceil(H * ceil(W/4) / 256), B).  Thread = 4 horizontally adjacent output pixels of one row, all three channels: the inverse map and
// the four bilinear taps are computed once per pixel and serve the three planes.  The source coordinate is evaluated in fp64 from the
// fp32 matrix (an fp32 coordinate near x = 640 is off by up to 3e-5 px, which a sharp image turns into a 3e-5 value error); the bilinear
// weights are fp32.  With the identity matrix the weights are exactly (1, 0, 0, 0) and the photometric terms below are exact, so a
// neutral augmenter returns its input bit for bit.
template <bool kNoise, bool kVec>
__global__ void __launch_bounds__(kAugThreads)
augment_images_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W, const float* __restrict__ inv, int tries,
                      const int32_t* __restrict__ pick, const float* __restrict__ photo, float noise_std, uint32_t k0, uint32_t k1) {
  const int b = blockIdx.y;
  const int wq = (W + 3) >> 2;
  const int t = blockIdx.x * kAugThreads + threadIdx.x;
  if (t >= wq * H) return;
  const int y = t / wq, xq = t - y * wq, x0 = xq << 2;
  const int p = __ldg(pick + b);
  double m00 = 1.0, m01 = 0.0, m02 = 0.0, m10 = 0.0, m11 = 1.0, m12 = 0.0;
  if (p >= 0) {
    const float* m = inv + ((size_t)b * tries + p) * 6;
    m00 = __ldg(m); m01 = __ldg(m + 1); m02 = __ldg(m + 2);
    m10 = __ldg(m + 3); m11 = __ldg(m + 4); m12 = __ldg(m + 5);
  }
  const size_t plane = (size_t)H * W;
  const float* src = in + (size_t)b * 3 * plane;
  const double xs_row = fma(m01, (double)y, m02), ys_row = fma(m11, (double)y, m12);
  float v[3][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    // clamped a little outside the image: every tap of a clamped coordinate is out of bounds, and the int conversion cannot overflow
    const double xs = fmin(fmax(fma(m00, (double)(x0 + j), xs_row), -2.0), (double)W + 1.0);
    const double ys = fmin(fmax(fma(m10, (double)(x0 + j), ys_row), -2.0), (double)H + 1.0);
    const double xf = floor(xs), yf = floor(ys);
    const int ix = (int)xf, iy = (int)yf;
    const float fx = (float)(xs - xf), fy = (float)(ys - yf);
    const float wx0 = 1.0f - fx, wy0 = 1.0f - fy;
    const float w_nw = wx0 * wy0, w_ne = fx * wy0, w_sw = wx0 * fy, w_se = fx * fy;
    const bool x0ok = (unsigned)ix < (unsigned)W, x1ok = (unsigned)(ix + 1) < (unsigned)W;
    const bool y0ok = (unsigned)iy < (unsigned)H, y1ok = (unsigned)(iy + 1) < (unsigned)H;
    const long long o = (long long)iy * W + ix;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float* s = src + ch * plane;
      const float a = (y0ok && x0ok) ? __ldg(s + o) : 0.f;
      const float bq = (y0ok && x1ok) ? __ldg(s + o + 1) : 0.f;
      const float c = (y1ok && x0ok) ? __ldg(s + o + W) : 0.f;
      const float d = (y1ok && x1ok) ? __ldg(s + o + W + 1) : 0.f;
      float r = w_nw * a;
      r = fmaf(w_ne, bq, r);
      r = fmaf(w_sw, c, r);
      v[ch][j] = fmaf(w_se, d, r);
    }
  }
  const float* ph = photo + (size_t)b * 5;
  const float contrast = __ldg(ph), beta = __ldg(ph + 1);
  // (v - 0.5)*c + 0.5 + beta as v*c + (0.5 - 0.5*c + beta): the same affine map, exact for c = 1, beta = 0
  const float shift = __fadd_rn(fmaf(-0.5f, contrast, 0.5f), beta);
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const float g = __ldg(ph + 2 + ch);
    float n[4] = {0.f, 0.f, 0.f, 0.f};
    if constexpr (kNoise) normals4((uint32_t)xq, (uint32_t)y, (uint32_t)ch, (uint32_t)b, k0, k1, n);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float r = __fmul_rn(fmaf(v[ch][j], contrast, shift), g);
      if constexpr (kNoise) r = fmaf(noise_std, n[j], r);
      v[ch][j] = fminf(fmaxf(r, 0.0f), 1.0f);
    }
    float* dst = out + ((size_t)b * 3 + ch) * plane + (size_t)y * W + x0;
    if constexpr (kVec) {
      *reinterpret_cast<float4*>(dst) = make_float4(v[ch][0], v[ch][1], v[ch][2], v[ch][3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (x0 + j < W) dst[j] = v[ch][j];
    }
  }
}

static bool overlaps(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
  const uintptr_t pa = reinterpret_cast<uintptr_t>(a), pb = reinterpret_cast<uintptr_t>(b);
  return pa < pb + b_bytes && pb < pa + a_bytes;
}

}  // namespace hk

extern "C" {

int hk_augment_pick(const float* fwd, int B, int tries, int K, int H, int W, const float* uv, float* uv_out, int32_t* pick,
                    void* stream) {
  using namespace hk;
  HK_REQUIRE(fwd && uv && uv_out && pick, "hk_augment_pick: null pointer");
  HK_REQUIRE(B > 0 && K > 0 && H > 0 && W > 0, "hk_augment_pick: bad shape");
  HK_REQUIRE(tries >= 1 && tries <= HK_AUGMENT_MAX_TRIES, "hk_augment_pick: tries must be in 1..%d", HK_AUGMENT_MAX_TRIES);
  const size_t uv_bytes = (size_t)B * K * 2 * sizeof(float);
  HK_REQUIRE(!overlaps(uv, uv_bytes, uv_out, uv_bytes), "hk_augment_pick: uv_out overlaps uv (in place is not supported)");
  const int threads = 128;
  augment_pick_kernel<<<ceil_div(B, threads), threads, 0, as_stream(stream)>>>(fwd, B, tries, K, (float)(W - 1), (float)(H - 1), uv,
                                                                                uv_out, pick);
  return check_launch("augment_pick_kernel");
}

int hk_augment_images(const float* in, float* out, int B, int H, int W, const float* inv, int tries, const int32_t* pick,
                      const float* photo, float noise_std, uint64_t key, void* stream) {
  using namespace hk;
  HK_REQUIRE(in && out && inv && pick && photo, "hk_augment_images: null pointer");
  HK_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "hk_augment_images: bad shape");
  HK_REQUIRE((long long)H * ((W + 3) / 4) + kAugThreads < (1LL << 31), "hk_augment_images: image too large");
  HK_REQUIRE(tries >= 1 && tries <= HK_AUGMENT_MAX_TRIES, "hk_augment_images: tries must be in 1..%d", HK_AUGMENT_MAX_TRIES);
  HK_REQUIRE(noise_std >= 0.f, "hk_augment_images: noise_std must be >= 0");
  const size_t bytes = (size_t)B * 3 * H * W * sizeof(float);
  HK_REQUIRE(!overlaps(in, bytes, out, bytes), "hk_augment_images: out overlaps in (in place is not supported)");
  const int per_image = H * ((W + 3) / 4);
  const dim3 grid(ceil_div(per_image, kAugThreads), B);
  const bool vec = (W & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  const uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
  cudaStream_t s = as_stream(stream);
#define HK_AUG_LAUNCH(NOISE, VEC) \
  augment_images_kernel<NOISE, VEC><<<grid, kAugThreads, 0, s>>>(in, out, H, W, inv, tries, pick, photo, noise_std, k0, k1)
  if (noise_std > 0.f) {
    if (vec) HK_AUG_LAUNCH(true, true); else HK_AUG_LAUNCH(true, false);
  } else {
    if (vec) HK_AUG_LAUNCH(false, true); else HK_AUG_LAUNCH(false, false);
  }
#undef HK_AUG_LAUNCH
  return check_launch("augment_images_kernel");
}

}  // extern "C"
