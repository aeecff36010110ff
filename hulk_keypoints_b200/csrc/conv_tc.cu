// tcgen05 implicit-GEMM convolution for sm_100a (SURVEY.md k2-k5): conv + folded-BN affine (+ residual) (+ ReLU).
//
// Replaces nn.Conv2d -> nn.BatchNorm2d(eval) -> (+= residual) -> nn.ReLU of BasicBlock.forward
// (reference src/resnet.py:56-67) and the 1x1 downsample (src/resnet.py:184-188), including the
// dilation-2 / dilation-4 stages of the output-stride-8 network (src/resnet.py:170-175,191-194).
//
// GEMM view: D[M = B*Ho*Wo, N = Cout] = A[M, K = kh*kw*Cin] * W[N, K]^T, bf16 operands, fp32 accumulate.
//   * A is never materialised.  Activations are NHWC bf16; a 4-D TMA tensor map (C, W, H, B) with a
//     (64 ch, 16 px, 4 rows, 1) box fetches, for filter tap (r, s), the input pixels of a 4x16 patch of OUTPUT
//     pixels shifted by (r*dil - pad, s*dil - pad); TMA zero-fills everything outside the image, which is
//     exactly the conv's zero padding.  With 128-byte swizzle the box lands in shared memory as 64 rows
//     x 128 B -- the canonical K-major SWIZZLE_128B UMMA operand.  Two boxes make one 128-row M tile, so
//     a 60x80 (or 120x160) feature map tiles exactly.  Stride-2 convs use the map's element strides.
//   * W is (Cout, kh*kw*Cin) bf16, K-major, fetched with a 2-D map (64 x BLOCK_N box).
//   * One K block = one tap x 64 channels.  tcgen05.mma (M=128, N=BLOCK_N, K=16) x4 per K block,
//     accumulators in TMEM, double-buffered (2 x BLOCK_N columns) so the epilogue of tile i overlaps the
//     MMAs of tile i+1.
//   * Warp roles (256 threads, 1 CTA/SM, persistent over tiles): warp0 = TMA producer (1 lane),
//     warp1 = MMA issuer (1 lane), warp2 = TMEM allocator, warps4-7 = epilogue (tcgen05.ld 32x32b,
//     fp32 scale/bias/residual/ReLU, bf16 NHWC store).
#include <cuda.h>

#include "hk_common.cuh"
#include "hk_ptx.cuh"

namespace hk {

constexpr int TC_BLOCK_M = 128;
constexpr int TC_BLOCK_K = 64;                          // bf16 elements = 128 bytes = one swizzle row
constexpr int TC_UMMA_K = 16;
constexpr int TC_BOX_H = 4, TC_BOX_W = 16;              // output pixels per TMA box (64)
constexpr int TC_BOX_PIX = TC_BOX_H * TC_BOX_W;
constexpr int TC_BOX_BYTES = TC_BOX_PIX * TC_BLOCK_K * 2;  // 8 KB
constexpr int TC_A_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;    // 16 KB
constexpr int TC_THREADS = 256;
constexpr int TC_EPI_WARP0 = 4;

struct ConvTcArgs {
  const float* scale;
  const float* bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* y;
  int B, Ho, Wo, Cout;
  int Cin, kh, kw, stride, pad, dil, relu;
  int tiles_x, tiles_per_img, num_boxes;
  int num_m_tiles, num_n_tiles, cblocks;
};

template <int BLOCK_N>
struct TcCfg {
  static constexpr int B_BYTES = BLOCK_N * TC_BLOCK_K * 2;
  static constexpr int STAGE_BYTES = TC_A_BYTES + B_BYTES;
  static constexpr int STAGES = (192 * 1024) / STAGE_BYTES > 8 ? 8 : (192 * 1024) / STAGE_BYTES;
  static constexpr int TMEM_COLS = 2 * BLOCK_N;  // 128 / 256 / 512: powers of two >= 32
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

__device__ __forceinline__ void tc_decode_box(const ConvTcArgs& a, int box, int& b, int& y0, int& x0) {
  if (box < a.num_boxes) {
    b = box / a.tiles_per_img;
    const int r = box - b * a.tiles_per_img;
    const int ty = r / a.tiles_x;
    y0 = ty * TC_BOX_H;
    x0 = (r - ty * a.tiles_x) * TC_BOX_W;
  } else {  // padding box of an odd tail: batch index out of range -> TMA zero fill, stores masked
    b = a.B;
    y0 = 0;
    x0 = 0;
  }
}

template <int BLOCK_N>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const ConvTcArgs a) {
  using Cfg = TcCfg<BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp: provably uniform
  const int total_tiles = a.num_m_tiles * a.num_n_tiles;
  const int num_kb = a.kh * a.kw * a.cblocks;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], 128);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_ptr_smem, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    {
      // ===================== TMA producer (whole warp waits, one elected lane issues) =====================
      uint32_t stage = 0, phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m_tile = tile / a.num_n_tiles, n_tile = tile - m_tile * a.num_n_tiles;
        int b0, y0, x0, b1, y1, x1;
        tc_decode_box(a, 2 * m_tile, b0, y0, x0);
        tc_decode_box(a, 2 * m_tile + 1, b1, y1, x1);
        for (int r = 0; r < a.kh; ++r) {
          for (int s = 0; s < a.kw; ++s) {
            const int dy = r * a.dil - a.pad, dx = s * a.dil - a.pad;
            const int kbase = (r * a.kw + s) * a.Cin;
            for (int cb = 0; cb < a.cblocks; ++cb) {
              ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 1);
              if (ptx::elect_one_sync()) {
                uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                ptx::mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                ptx::tma_load_4d(sa, &map_x, &full_bar[stage], cb * TC_BLOCK_K, x0 * a.stride + dx, y0 * a.stride + dy, b0);
                ptx::tma_load_4d(sa + TC_BOX_BYTES, &map_x, &full_bar[stage], cb * TC_BLOCK_K, x1 * a.stride + dx,
                                 y1 * a.stride + dy, b1);
                ptx::tma_load_2d(sa + TC_A_BYTES, &map_w, &full_bar[stage], kbase + cb * TC_BLOCK_K, n_tile * BLOCK_N);
              }
              __syncwarp();
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer (whole warp waits, one elected lane issues) =====================
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(TC_BLOCK_M, BLOCK_N);
      uint32_t stage = 0, phase = 0, it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, 2);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase, 3);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t adesc = ptx::make_smem_desc_sw128(sa);
          const uint64_t bdesc = ptx::make_smem_desc_sw128(sa + TC_A_BYTES);
          if (ptx::elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k) {
              // advance 16 bf16 = 32 bytes along K inside the swizzle row: +2 in the (addr >> 4) field
              ptx::umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            ptx::umma_commit(&empty_bar[stage]);                         // frees the smem slot when the MMAs retire
            if (kb == num_kb - 1) ptx::umma_commit(&tmem_full_bar[acc]);  // accumulator ready for the epilogue
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= TC_EPI_WARP0) {
    // ===================== epilogue =====================
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const int py = (row & 63) >> 4, px = row & 15;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const int m_tile = tile / a.num_n_tiles, n_tile = tile - m_tile * a.num_n_tiles;
      int b, y0, x0;
      tc_decode_box(a, 2 * m_tile + (row >> 6), b, y0, x0);
      const int oy = y0 + py, ox = x0 + px;
      const bool valid = (b < a.B) && (oy < a.Ho) && (ox < a.Wo);
      const size_t off = valid ? (((size_t)b * a.Ho + oy) * a.Wo + ox) * a.Cout + (size_t)n_tile * BLOCK_N : 0;
      const float* scale = a.scale + n_tile * BLOCK_N;
      const float* bias = a.bias + n_tile * BLOCK_N;

      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase, 4);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        uint32_t r[32];
        ptx::tmem_ld_32x32(taddr + c0, r);
        ptx::tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int c = c0 + g * 8;
            const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale + c));
            const float4 s1 = __ldg(reinterpret_cast<const float4*>(scale + c + 4));
            const float4 t0 = __ldg(reinterpret_cast<const float4*>(bias + c));
            const float4 t1 = __ldg(reinterpret_cast<const float4*>(bias + c + 4));
            float v[8];
            v[0] = fmaf(__uint_as_float(r[g * 8 + 0]), s0.x, t0.x);
            v[1] = fmaf(__uint_as_float(r[g * 8 + 1]), s0.y, t0.y);
            v[2] = fmaf(__uint_as_float(r[g * 8 + 2]), s0.z, t0.z);
            v[3] = fmaf(__uint_as_float(r[g * 8 + 3]), s0.w, t0.w);
            v[4] = fmaf(__uint_as_float(r[g * 8 + 4]), s1.x, t1.x);
            v[5] = fmaf(__uint_as_float(r[g * 8 + 5]), s1.y, t1.y);
            v[6] = fmaf(__uint_as_float(r[g * 8 + 6]), s1.z, t1.z);
            v[7] = fmaf(__uint_as_float(r[g * 8 + 7]), s1.w, t1.w);
            if (a.residual) {
              const uint4 rq = __ldg(reinterpret_cast<const uint4*>(a.residual + off + c));
              float lo, hi;
              unpack_bf16x2(rq.x, lo, hi); v[0] += lo; v[1] += hi;
              unpack_bf16x2(rq.y, lo, hi); v[2] += lo; v[3] += hi;
              unpack_bf16x2(rq.z, lo, hi); v[4] += lo; v[5] += hi;
              unpack_bf16x2(rq.w, lo, hi); v[6] += lo; v[7] += hi;
            }
            if (a.relu) {
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            *reinterpret_cast<uint4*>(a.y + off + c) =
                make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          }
        }
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(&tmem_empty_bar[acc]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ---------------- host side ----------------
template <int BLOCK_N>
static int launch_tc(const CUtensorMap& mx, const CUtensorMap& mw, const ConvTcArgs& a, cudaStream_t s) {
  using Cfg = TcCfg<BLOCK_N>;
  if (int rc = opt_in_smem<conv_tc_kernel<BLOCK_N>>(Cfg::SMEM_BYTES, "conv(tcgen05)")) return rc;
  const int total = a.num_m_tiles * a.num_n_tiles;
  int grid = sm_count();
  if (grid > total) grid = total;
  conv_tc_kernel<BLOCK_N><<<grid, TC_THREADS, Cfg::SMEM_BYTES, s>>>(mx, mw, a);
  return check_launch("conv_tc_kernel");
}

bool conv_tc2_applicable(const HkConvDesc& d);
int conv_tc2_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                    const void* residual, void* y, void* bn_acc, cudaStream_t s);
bool conv_tc2h_applicable(const HkConvDesc& d);
int conv_tc2h_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                     const void* residual, void* y, void* bn_acc, cudaStream_t s);
bool conv_tc_c64_applicable(const HkConvDesc& d);
int conv_tc_c64_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                       const void* residual, void* y, void* bn_acc, cudaStream_t s);

// bn_acc != nullptr: the epilogue also adds per-channel sum y / sum y^2 of the stored outputs to the accumulators (train-mode BatchNorm
// statistics; specialised kernels only -- *stats_done tells the caller whether it still has to run the stand-alone reduction)
int conv_tc_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                   const void* residual, void* y, cudaStream_t s, void* bn_acc = nullptr, bool* stats_done = nullptr) {
  if (stats_done) *stats_done = false;
  HK_REQUIRE(d.in_dtype == HK_BF16 && d.out_dtype == HK_BF16 && !d.in_is_nchw, "conv(tcgen05): needs NHWC bf16 in and out");
  HK_REQUIRE(d.in_c % TC_BLOCK_K == 0, "conv(tcgen05): in_c=%d must be a multiple of 64", d.in_c);
  HK_REQUIRE(d.out_c % 64 == 0, "conv(tcgen05): out_c=%d must be a multiple of 64", d.out_c);
  HK_REQUIRE(d.stride == 1 || d.stride == 2, "conv(tcgen05): stride must be 1 or 2");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(residual) & 15) == 0,
             "conv(tcgen05): buffers must be 16-byte aligned");

  // layer1 shape (3x3, 64 -> 64, stride 1): resident weights + haloed boxes, 3.6x less L2->SM traffic
  const bool specialised = d.algo != HK_CONV_TCGEN05_1CTA;
  if (stats_done) *stats_done = bn_acc && specialised && (conv_tc_c64_applicable(d) || conv_tc2_applicable(d));
  if (specialised && conv_tc_c64_applicable(d)) return conv_tc_c64_launch(d, x, w, scale, bias, residual, y, bn_acc, s);
  // operand-traffic-bound 3x3 shapes: CTA-pair kernel with one haloed activation box per horizontal tap
  if (specialised && conv_tc2_applicable(d) && conv_tc2h_applicable(d)) return conv_tc2h_launch(d, x, w, scale, bias, residual, y, bn_acc, s);
  // Cout >= 128: CTA-pair kernel (cta_group::2, M=256), half the weight tile per SM
  if (specialised && conv_tc2_applicable(d)) return conv_tc2_launch(d, x, w, scale, bias, residual, y, bn_acc, s);

  const int block_n = d.out_c % 256 == 0 ? 256 : (d.out_c % 128 == 0 ? 128 : 64);
  const int ktot = d.kh * d.kw * d.in_c;

  const char* who = "conv(tcgen05)";
  CUtensorMap mx, mw;
  if (int rc = tmap_nhwc_bf16(&mx, x, d.batch, d.in_h, d.in_w, d.in_c, TC_BOX_W, TC_BOX_H, d.stride, who, "activations")) return rc;
  if (int rc = tmap_kmajor_bf16(&mw, w, ktot, d.out_c, block_n, who, "weights")) return rc;

  ConvTcArgs a;
  a.scale = scale; a.bias = bias;
  a.residual = static_cast<const __nv_bfloat16*>(residual);
  a.y = static_cast<__nv_bfloat16*>(y);
  a.B = d.batch; a.Ho = d.out_h; a.Wo = d.out_w; a.Cout = d.out_c;
  a.Cin = d.in_c; a.kh = d.kh; a.kw = d.kw; a.stride = d.stride; a.pad = d.pad; a.dil = d.dil; a.relu = d.relu;
  a.tiles_x = ceil_div(d.out_w, TC_BOX_W);
  a.tiles_per_img = a.tiles_x * ceil_div(d.out_h, TC_BOX_H);
  const long long boxes = (long long)a.tiles_per_img * d.batch;
  HK_REQUIRE(boxes < 0x3fffffffLL, "conv(tcgen05): too many tiles");
  a.num_boxes = (int)boxes;
  a.num_m_tiles = (a.num_boxes + 1) / 2;
  a.num_n_tiles = d.out_c / block_n;
  a.cblocks = d.in_c / TC_BLOCK_K;
  switch (block_n) {
    case 256: return launch_tc<256>(mx, mw, a, s);
    case 128: return launch_tc<128>(mx, mw, a, s);
    default: return launch_tc<64>(mx, mw, a, s);
  }
}

int conv_ffma_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                     const void* residual, void* y, cudaStream_t s);

}  // namespace hk

extern "C" int hk_conv_bn_act_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale,
                                  const float* bias, const void* residual_or_null, void* y, void* stream) {
  using namespace hk;
  HK_REQUIRE(desc && x && w_packed && scale && bias && y, "hk_conv_bn_act_fwd: null pointer");
  const HkConvDesc& d = *desc;
  HK_REQUIRE(d.batch > 0 && d.in_h > 0 && d.in_w > 0 && d.in_c > 0 && d.out_c > 0 && d.kh > 0 && d.kw > 0 && d.stride > 0 &&
                 d.dil > 0 && d.pad >= 0,
             "hk_conv_bn_act_fwd: bad descriptor");
  const int eh = d.dil * (d.kh - 1) + 1, ew = d.dil * (d.kw - 1) + 1;
  HK_REQUIRE(d.in_h + 2 * d.pad >= eh && d.in_w + 2 * d.pad >= ew, "hk_conv_bn_act_fwd: kernel larger than padded input");
  HK_REQUIRE(d.out_h == (d.in_h + 2 * d.pad - eh) / d.stride + 1 && d.out_w == (d.in_w + 2 * d.pad - ew) / d.stride + 1,
             "hk_conv_bn_act_fwd: out_h/out_w (%d,%d) inconsistent with the descriptor", d.out_h, d.out_w);
  if (d.algo == HK_CONV_TCGEN05 || d.algo == HK_CONV_TCGEN05_1CTA) return conv_tc_launch(d, x, w_packed, scale, bias, residual_or_null, y, as_stream(stream));
  if (d.algo == HK_CONV_FFMA) return conv_ffma_launch(d, x, w_packed, scale, bias, residual_or_null, y, as_stream(stream));
  return fail(HK_ERR_BAD_ARG, "hk_conv_bn_act_fwd: unknown algo %d", d.algo);
}

// Train-mode forward of one conv + the statistics pass of its BatchNorm: y = conv(x) (raw: the caller passes scale = 1, bias = 0) and
// acc += per-channel (sum y, sum y^2) of the bf16 values stored, gathered in the conv epilogue (hk_bn_acc.cuh) -- the activation is not
// read again for its statistics.  Shapes outside the specialised tcgen05 kernels run the conv and then hk_bn_stats_acc (two launches).
extern "C" int hk_bn_stats_acc(const void* y, long long P, int C, void* acc, void* stream);
extern "C" int hk_conv_bn_stats_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale, const float* bias,
                                    void* y, void* acc, void* stream) {
  using namespace hk;
  HK_REQUIRE(desc && x && w_packed && scale && bias && y && acc, "hk_conv_bn_stats_fwd: null pointer");
  const HkConvDesc& d = *desc;
  HK_REQUIRE(d.algo == HK_CONV_TCGEN05 && d.in_dtype == HK_BF16 && d.out_dtype == HK_BF16 && !d.in_is_nchw && !d.relu,
             "hk_conv_bn_stats_fwd: tcgen05 path only (NHWC bf16 in and out, no ReLU: BatchNorm sees the raw conv output)");
  HK_REQUIRE(d.batch > 0 && d.in_h > 0 && d.in_w > 0 && d.in_c > 0 && d.out_c > 0 && d.kh > 0 && d.kw > 0 && d.stride > 0 && d.dil > 0 && d.pad >= 0,
             "hk_conv_bn_stats_fwd: bad descriptor");
  const int eh = d.dil * (d.kh - 1) + 1, ew = d.dil * (d.kw - 1) + 1;
  HK_REQUIRE(d.out_h == (d.in_h + 2 * d.pad - eh) / d.stride + 1 && d.out_w == (d.in_w + 2 * d.pad - ew) / d.stride + 1,
             "hk_conv_bn_stats_fwd: out_h/out_w (%d,%d) inconsistent with the descriptor", d.out_h, d.out_w);
  HK_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 31) == 0, "hk_conv_bn_stats_fwd: accumulators must be 32-byte aligned");
  bool done = false;
  int rc = conv_tc_launch(d, x, w_packed, scale, bias, nullptr, y, as_stream(stream), acc, &done);
  if (rc || done) return rc;
  return hk_bn_stats_acc(y, (long long)d.batch * d.out_h * d.out_w, d.out_c, acc, stream);
}
