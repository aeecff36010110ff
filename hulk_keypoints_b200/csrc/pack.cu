// Weight repack: OIHW fp32 state_dict tensor -> O(HW)I ("KRSC") fp32/bf16 GEMM-B operand, and
// BatchNorm(eval) -> per-channel (scale, bias) applied in the conv epilogue.
//
// The reference keeps nn.Conv2d weights as (cout, cin, kh, kw) and applies nn.BatchNorm2d as a separate
// op (src/resnet.py:46,49,139,187).  In eval() that op is y = (x - mean) / sqrt(var + eps) * gamma + beta,
// i.e. y = x * scale + bias with scale = gamma / sqrt(var + eps), bias = beta - mean * scale.  The scale is
// kept OUT of the weights (applied to the fp32 accumulator) so bf16 weight rounding is not perturbed.
#include "hk_common.cuh"

namespace hk {

template <typename OutT>
__global__ void __launch_bounds__(256)
pack_weights_kernel(const float* __restrict__ w_oihw, OutT* __restrict__ w_out, int cout, int cin, int khw) {
  const long long total = (long long)cout * cin * khw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    // destination index: ((o * khw + t) * cin + c)
    const int c = (int)(i % cin);
    const long long r = i / cin;
    const int t = (int)(r % khw);
    const int o = (int)(r / khw);
    const float v = __ldg(w_oihw + ((size_t)o * cin + c) * khw + t);
    store_from_float<OutT>(w_out + i, v);
  }
}

// Data-gradient weights: dX = conv(dY, W') with W'[ci, r', s', co] = W[co, ci, kh-1-r', kw-1-s'] (taps flipped, channel roles
// swapped); same pad/dilation as the forward conv when pad == dil*(k-1)/2 (every conv of this network).
__global__ void __launch_bounds__(256)
pack_weights_dgrad_kernel(const float* __restrict__ w_oihw, __nv_bfloat16* __restrict__ w_out, int cout, int cin, int kh, int kw) {
  const int khw = kh * kw;
  const long long total = (long long)cout * cin * khw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    // destination index: ((ci * khw + t') * cout + co)
    const int co = (int)(i % cout);
    const long long r = i / cout;
    const int t = (int)(r % khw);
    const int ci = (int)(r / khw);
    w_out[i] = __float2bfloat16_rn(__ldg(w_oihw + ((size_t)co * cin + ci) * khw + (khw - 1 - t)));
  }
}

// All convolutions of the network in ONE launch (training repacks the weights every step): blockIdx.y = item, the x index space of an
// item is [0, n) for the forward layout (cout, khw, cin) followed by [n, 2n) for the data-gradient layout (cin, khw flipped, cout).
__global__ void __launch_bounds__(256) pack_weights_many_kernel(const HkPackItem* __restrict__ items) {
  const HkPackItem it = items[blockIdx.y];
  const long long n = (long long)it.cout * it.cin * it.khw;
  const long long total = it.w_dgrad ? 2 * n : n;
  const float* __restrict__ w = it.w;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (i < n) {
      const int c = (int)(i % it.cin);
      const long long r = i / it.cin;
      const int t = (int)(r % it.khw);
      const int o = (int)(r / it.khw);
      static_cast<__nv_bfloat16*>(it.w_fwd)[i] = __float2bfloat16_rn(__ldg(w + ((size_t)o * it.cin + c) * it.khw + t));
    } else {
      const long long j = i - n;
      const int co = (int)(j % it.cout);
      const long long r = j / it.cout;
      const int t = (int)(r % it.khw);
      const int ci = (int)(r / it.khw);
      static_cast<__nv_bfloat16*>(it.w_dgrad)[j] = __float2bfloat16_rn(__ldg(w + ((size_t)co * it.cin + ci) * it.khw + (it.khw - 1 - t)));
    }
  }
}

// The same through a shared-memory tile (round 2): the element-wise kernel above gathers its source at a 36-byte stride (8x read
// amplification) and writes the data-gradient layout 2 bytes at a time: 167 us per step for 87 MB of weights, ~90 us of it exposed at
// per-GPU batch 4 (the first block conv waits for the packed weights).  Here a CTA loads 64 output channels x 32 input channels x khw taps
// as 64 contiguous runs, then writes both layouts in 64-byte runs: forward (co, t, ci0..ci0+31), data gradient (ci, t', co0..co0+63); the
// tile pitch is odd, so the strided shared-memory reads of both passes are conflict-free.  blockIdx.y = item, blockIdx.x strides over the
// item's tiles.  Needs cout % 64 == 0 and cin % 32 == 0 for every item (all block convs of the backbone).
constexpr int PK_CO = 64, PK_CI = 32;
__global__ void __launch_bounds__(256) pack_weights_many_tiled_kernel(const HkPackItem* __restrict__ items) {
  extern __shared__ float pk_tile[];   // [64][32*khw + 1]
  const HkPackItem it = items[blockIdx.y];
  const int khw = it.khw, row = PK_CI * khw, pitch = row | 1;
  const int tiles_ci = it.cin / PK_CI, ntiles = (it.cout / PK_CO) * tiles_ci;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const float* __restrict__ w = it.w;
  __nv_bfloat16* __restrict__ out_f = static_cast<__nv_bfloat16*>(it.w_fwd);
  __nv_bfloat16* __restrict__ out_d = static_cast<__nv_bfloat16*>(it.w_dgrad);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int co0 = (tile / tiles_ci) * PK_CO, ci0 = (tile % tiles_ci) * PK_CI;
    for (int r = wid; r < PK_CO; r += 8) {
      const float* src = w + ((size_t)(co0 + r) * it.cin + ci0) * khw;   // `row` contiguous floats
      for (int c = lane; c < row; c += 32) pk_tile[r * pitch + c] = __ldg(src + c);
    }
    __syncthreads();
    for (int r = wid; r < PK_CO; r += 8) {         // forward layout (co, t, ci): lane = ci
      for (int t = 0; t < khw; ++t)
        out_f[((size_t)(co0 + r) * khw + t) * it.cin + ci0 + lane] = __float2bfloat16_rn(pk_tile[r * pitch + lane * khw + t]);
    }
    if (out_d) {                                    // data-gradient layout (ci, t', co) with flipped taps: lane = co (two halves)
      for (int ci = wid; ci < PK_CI; ci += 8) {
        for (int t = 0; t < khw; ++t) {
          __nv_bfloat16* dst = out_d + ((size_t)(ci0 + ci) * khw + t) * it.cout + co0;
          dst[lane] = __float2bfloat16_rn(pk_tile[lane * pitch + ci * khw + (khw - 1 - t)]);
          dst[lane + 32] = __float2bfloat16_rn(pk_tile[(lane + 32) * pitch + ci * khw + (khw - 1 - t)]);
        }
      }
    }
    __syncthreads();
  }
}

__global__ void bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                               const float* __restrict__ var, float eps, int cout, float* __restrict__ scale,
                               float* __restrict__ bias) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout) return;
  if (gamma) {
    // same op order as ATen's eval batch_norm: invstd = 1/sqrt(var+eps); w*invstd; b - mean*w*invstd
    const float invstd = 1.0f / sqrtf(var[i] + eps);
    const float s = gamma[i] * invstd;
    scale[i] = s;
    bias[i] = beta[i] - mean[i] * s;
  } else {
    scale[i] = 1.0f;
    bias[i] = 0.0f;
  }
}

}  // namespace hk

extern "C" int hk_pack_conv_weights(const float* w_oihw, const float* bn_gamma, const float* bn_beta, const float* bn_mean,
                                    const float* bn_var, float bn_eps, int cout, int cin, int kh, int kw, int w_dtype,
                                    void* w_out, float* scale_out, float* bias_out, void* stream) {
  using namespace hk;
  HK_REQUIRE(w_oihw && w_out && scale_out && bias_out, "hk_pack_conv_weights: null pointer");
  HK_REQUIRE(cout > 0 && cin > 0 && kh > 0 && kw > 0, "hk_pack_conv_weights: bad shape");
  const bool all = bn_gamma && bn_beta && bn_mean && bn_var;
  const bool none = !bn_gamma && !bn_beta && !bn_mean && !bn_var;
  HK_REQUIRE(all || none, "hk_pack_conv_weights: pass all four BatchNorm vectors or none");
  HK_REQUIRE(w_dtype == HK_BF16 || w_dtype == HK_F32, "hk_pack_conv_weights: w_dtype must be bf16 or f32");
  cudaStream_t s = as_stream(stream);
  const long long total = (long long)cout * cin * kh * kw;
  int blocks = (int)ceil_div_ll(total, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (w_dtype == HK_BF16)
    pack_weights_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(w_oihw, static_cast<__nv_bfloat16*>(w_out), cout, cin, kh * kw);
  else
    pack_weights_kernel<float><<<blocks, 256, 0, s>>>(w_oihw, static_cast<float*>(w_out), cout, cin, kh * kw);
  int rc = check_launch("pack_weights_kernel");
  if (rc) return rc;
  bn_fold_kernel<<<ceil_div(cout, 128), 128, 0, s>>>(bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, cout, scale_out, bias_out);
  return check_launch("bn_fold_kernel");
}

extern "C" int hk_pack_conv_weights_dgrad(const float* w_oihw, int cout, int cin, int kh, int kw, void* w_out, void* stream) {
  using namespace hk;
  HK_REQUIRE(w_oihw && w_out, "hk_pack_conv_weights_dgrad: null pointer");
  HK_REQUIRE(cout > 0 && cin > 0 && kh > 0 && kw > 0, "hk_pack_conv_weights_dgrad: bad shape");
  const long long total = (long long)cout * cin * kh * kw;
  int blocks = (int)ceil_div_ll(total, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  pack_weights_dgrad_kernel<<<blocks, 256, 0, as_stream(stream)>>>(w_oihw, static_cast<__nv_bfloat16*>(w_out), cout, cin, kh, kw);
  return check_launch("pack_weights_dgrad_kernel");
}

extern "C" int hk_pack_conv_weights_many(const HkPackItem* items_dev, int n_items, long long max_elems, void* stream) {
  using namespace hk;
  HK_REQUIRE(items_dev && n_items > 0 && max_elems > 0, "hk_pack_conv_weights_many: bad argument");
  long long bx = ceil_div_ll(2 * max_elems, 256 * 8);  // 8 elements per thread for the largest item
  if (bx > 1024) bx = 1024;
  if (bx < 1) bx = 1;
  pack_weights_many_kernel<<<dim3((unsigned)bx, (unsigned)n_items), 256, 0, as_stream(stream)>>>(items_dev);
  return check_launch("pack_weights_many_kernel");
}

// Tiled variant of hk_pack_conv_weights_many (see pack_weights_many_tiled_kernel): every item must have cout % 64 == 0, cin % 32 == 0 and
// khw <= max_khw (the caller checks; the shared-memory tile is sized by max_khw).
extern "C" int hk_pack_conv_weights_many_tiled(const HkPackItem* items_dev, int n_items, int max_khw, long long max_elems, void* stream) {
  using namespace hk;
  HK_REQUIRE(items_dev && n_items > 0 && max_khw > 0 && max_khw <= 25 && max_elems > 0, "hk_pack_conv_weights_many_tiled: bad argument");
  const int smem = PK_CO * ((PK_CI * max_khw) | 1) * (int)sizeof(float);
  if (int rc = opt_in_smem<pack_weights_many_tiled_kernel>(smem, "hk_pack_conv_weights_many_tiled")) return rc;
  long long bx = ceil_div_ll(max_elems, (long long)PK_CO * PK_CI * max_khw);   // tiles of the largest item
  if (bx > 64) bx = 64;
  if (bx < 1) bx = 1;
  pack_weights_many_tiled_kernel<<<dim3((unsigned)bx, (unsigned)n_items), 256, smem, as_stream(stream)>>>(items_dev);
  return check_launch("pack_weights_many_tiled_kernel");
}
