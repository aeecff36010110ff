// tcgen05 weight-gradient ("wgrad") implicit GEMM for the backbone convolutions (SURVEY.md §8 f1, k14).
//
// Autograd of nn.Conv2d (reference src/resnet.py:36,185 as trained by train.py:35):
//   dW[co, ci, r, s] = sum_{b,oy,ox} dY[b,oy,ox,co] * X[b, oy*stride - pad + r*dil, ox*stride - pad + s*dil, ci]
// GEMM view per filter tap (r,s):  D[M = Cout, N = Cin] = dY^T[Cout, P] * X_shifted[P, Cin], the reduction runs over the
// P = B*Ho*Wo output pixels.  Both operands are NHWC activations, i.e. the GEMM-K dimension (pixels) is the STRIDED one:
//   * the same 4-D TMA boxes as the forward kernel -- (64 ch, 16 px, 4 rows) with SWIZZLE_128B, tap shift / zero padding /
//     stride-2 element strides done by the tensor map -- land in shared memory as [64 pixels][64 channels];
//   * that tile is fed to tcgen05.mma as an MN-MAJOR operand (instruction-descriptor bits 15/16; canonical layout
//     ((8,n),(8,k)) x 16 B: 64 channels contiguous, 8-pixel groups 1024 B apart (SBO), 64-channel groups one box apart
//     (LBO)), so no transpose pass over dY or X ever touches HBM;
//   * one pipeline stage = 64 pixels = 4 MMAs (K = 16 pixels = 2048 B further down the tile).
// Work unit = (K split, tap, 128-row Cout tile, BLOCK_N-column Cin tile); units are distributed round-robin over one
// persistent CTA per SM; fp32 accumulators in TMEM (double-buffered), written as fp32 partials [split][Cout][tap][Cin] and
// summed in a fixed order by wgrad_reduce_kernel into the OIHW fp32 gradient -- deterministic, no atomics.
#include <cuda.h>
#include <stdlib.h>

#include "hk_common.cuh"
#include "hk_ptx.cuh"

namespace hk {

constexpr int WG_THREADS = 256;
constexpr int WG_BOX_H = 4, WG_BOX_W = 16;
constexpr int WG_BOX_BYTES = 64 * 128;  // 64 pixels x 64 channels bf16
constexpr int WG_A_BYTES = 2 * WG_BOX_BYTES;

struct WgradArgs {
  float* ws;
  int B, Ho, Wo, Cout, Cin, kh, kw, stride, pad, dil;
  int tiles_x, tiles_per_img, num_boxes;
  int m_tiles, n_tiles, taps, ksplit, boxes_per_split;
  int cout64;  // Cout == 64: the single 64-channel dY box is loaded twice (rows 64..127 of the accumulator are ignored) ...
  int tap_pairs;  // ... or, stride 1: TWO taps per unit.  dW_t[co,ci] = sum_p dY[p,co] X[p+off_t,ci] = sum_q dY[q-off_t,co] X[q,ci]: the shift moves
                  // to dY, rows 0..63 of the A operand are dY shifted for tap 2u and rows 64..127 dY shifted for tap 2u+1, B is the unshifted X
                  // box -- all 128 accumulator rows do useful work (5 units instead of 9 per K split for a 3x3 conv)
  int tap_units;  // units along the tap axis: taps, or ceil(taps / 2) with tap_pairs
};

template <int BLOCK_N>
struct WgCfg {
  static constexpr int B_BYTES = (BLOCK_N / 64) * WG_BOX_BYTES;
  static constexpr int STAGE_BYTES = WG_A_BYTES + B_BYTES;
  static constexpr int STAGES = (192 * 1024) / STAGE_BYTES > 8 ? 8 : (192 * 1024) / STAGE_BYTES;
  static constexpr int TMEM_COLS = 2 * BLOCK_N < 32 ? 32 : 2 * BLOCK_N;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
};

// MN-major, SWIZZLE_128B shared-memory descriptor: LBO = distance between 64-element groups along M/N (one TMA box),
// SBO = distance between 8-row groups along K (1024 B)
__device__ __forceinline__ uint64_t make_smem_desc_mn_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(WG_BOX_BYTES >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__device__ __forceinline__ void wg_decode_unit(const WgradArgs& a, int u, int& ks, int& tap, int& m, int& n) {
  n = u % a.n_tiles;
  u /= a.n_tiles;
  m = u % a.m_tiles;
  u /= a.m_tiles;
  tap = u % a.tap_units;
  ks = u / a.tap_units;
}
__device__ __forceinline__ void wg_decode_box(const WgradArgs& a, int box, int& b, int& y0, int& x0) {
  b = box / a.tiles_per_img;
  const int r = box - b * a.tiles_per_img;
  const int ty = r / a.tiles_x;
  y0 = ty * WG_BOX_H;
  x0 = (r - ty * a.tiles_x) * WG_BOX_W;
}

template <int BLOCK_N>
__global__ void __launch_bounds__(WG_THREADS, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x, const WgradArgs a) {
  using Cfg = WgCfg<BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int total_units = a.ksplit * a.tap_units * a.m_tiles * a.n_tiles;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_dy);
    ptx::prefetch_tensormap(&map_x);
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
    // ===================== TMA producer (whole warp waits, one elected lane issues) =====================
    uint32_t stage = 0, phase = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
      int ks, tap, m, n;
      wg_decode_unit(a, u, ks, tap, m, n);
      // tap_pairs: `tap` is a pair index; the two taps' shifts go to the two dY boxes, X stays put
      const int t0 = a.tap_pairs ? 2 * tap : tap, t1 = a.tap_pairs ? min(2 * tap + 1, a.taps - 1) : tap;
      const int r = t0 / a.kw, s = t0 - r * a.kw;
      const int dy = r * a.dil - a.pad, dx = s * a.dil - a.pad;
      const int r1 = t1 / a.kw, s1 = t1 - r1 * a.kw;
      const int dy1 = r1 * a.dil - a.pad, dx1 = s1 * a.dil - a.pad;
      const int ax0 = a.tap_pairs ? -dx : 0, ay0 = a.tap_pairs ? -dy : 0, ax1 = a.tap_pairs ? -dx1 : 0, ay1 = a.tap_pairs ? -dy1 : 0;
      const int bdx = a.tap_pairs ? 0 : dx, bdy = a.tap_pairs ? 0 : dy;
      const int box_lo = ks * a.boxes_per_split;
      const int box_hi = min(box_lo + a.boxes_per_split, a.num_boxes);
      const int co0 = m * 128, co1 = a.cout64 ? 0 : co0 + 64;
      for (int box = box_lo; box < box_hi; ++box) {
        int b, y0, x0;
        wg_decode_box(a, box, b, y0, x0);
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 41);
        if (ptx::elect_one_sync()) {
          uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
          ptx::mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
          ptx::tma_load_4d(sa, &map_dy, &full_bar[stage], co0, x0 + ax0, y0 + ay0, b);
          ptx::tma_load_4d(sa + WG_BOX_BYTES, &map_dy, &full_bar[stage], co1, x0 + ax1, y0 + ay1, b);
#pragma unroll
          for (int j = 0; j < BLOCK_N / 64; ++j)
            ptx::tma_load_4d(sa + WG_A_BYTES + j * WG_BOX_BYTES, &map_x, &full_bar[stage], n * BLOCK_N + j * 64, x0 * a.stride + bdx,
                             y0 * a.stride + bdy, b);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp waits, one elected lane issues) =====================
    constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, BLOCK_N) | (1u << 15) | (1u << 16);  // A and B MN-major
    uint32_t stage = 0, phase = 0, it = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const int ks = u / (a.tap_units * a.m_tiles * a.n_tiles);
      const int box_lo = ks * a.boxes_per_split;
      const int nbox = min(box_lo + a.boxes_per_split, a.num_boxes) - box_lo;
      ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, 42);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
      for (int kb = 0; kb < nbox; ++kb) {
        ptx::mbar_wait(&full_bar[stage], phase, 43);
        ptx::tc_fence_after();
        const uint32_t sa = ptx::smem_u32(smem + stage * Cfg::STAGE_BYTES);
        if (ptx::elect_one_sync()) {
          const uint64_t adesc = make_smem_desc_mn_sw128(sa);
          const uint64_t bdesc = make_smem_desc_mn_sw128(sa + WG_A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k)  // 16 pixels = 2048 bytes further along K: +128 in the (addr >> 4) field
            ptx::umma_bf16(d_tmem, adesc + 128 * k, bdesc + 128 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          ptx::umma_commit(&empty_bar[stage]);
          if (kb == nbox - 1) ptx::umma_commit(&tmem_full_bar[acc]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: TMEM -> fp32 partial tile in the workspace =====================
    const int q = warp & 3;
    const int row = q * 32 + lane;  // accumulator row = output channel within the 128-row tile
    uint32_t it = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      int ks, tap, m, n;
      wg_decode_unit(a, u, ks, tap, m, n);
      int co = m * 128 + row;
      bool valid = co < a.Cout && !(a.cout64 && row >= 64);
      if (a.tap_pairs) {   // rows 0..63: tap 2u, rows 64..127: tap 2u+1 (absent for the last unit of an odd tap count)
        const int second = row >> 6;
        co = row & 63;
        tap = 2 * tap + second;
        valid = tap < a.taps;
      }
      float* dst = a.ws + (((size_t)ks * a.Cout + co) * a.taps + (valid ? tap : 0)) * a.Cin + (size_t)n * BLOCK_N;
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase, 44);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        uint32_t r[32];
        ptx::tmem_ld_32x32(taddr + c0, r);
        ptx::tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int g = 0; g < 8; ++g)
            *reinterpret_cast<float4*>(dst + c0 + g * 4) = make_float4(__uint_as_float(r[g * 4]), __uint_as_float(r[g * 4 + 1]),
                                                                        __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3]));
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

// dw[co][ci][tap] (+)= sum_ks ws[ks][co][tap][ci]; thread index runs in workspace order (coalesced reads; the 4-byte writes at a
// 36-byte stride are merged in L2).  A block-per-(co, ci chunk) version that transposes through shared memory for coalesced writes was
// measured 0.25-0.35 ms per step SLOWER (fewer loads in flight per SM) and dropped.
// Four consecutive input channels per thread (one 16-byte load per split, four splits in flight); the sum runs over the splits in
// ascending order, as before.
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ ws, float* __restrict__ dw, int ksplit, int Cout, int taps,
                                                          int Cin, int accumulate) {
  const long long total4 = (long long)Cout * taps * Cin / 4;
  const float4* ws4 = reinterpret_cast<const float4*>(ws);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int k = 0;
    for (; k + 4 <= ksplit; k += 4) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldcs(ws4 + (size_t)(k + u) * total4 + i);
#pragma unroll
      for (int u = 0; u < 4; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
    for (; k < ksplit; ++k) {
      const float4 v = __ldcs(ws4 + (size_t)k * total4 + i);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    const long long e = i * 4;
    const int ci = (int)(e % Cin);
    const long long r = e / Cin;
    const int tap = (int)(r % taps);
    const int co = (int)(r / taps);
    float* dst = dw + ((size_t)co * Cin + ci) * taps + tap;
    const float sv[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) dst[(size_t)j * taps] = (accumulate ? dst[(size_t)j * taps] : 0.f) + sv[j];
  }
}

struct WgradPlan {
  int block_n, m_tiles, n_tiles, taps, ksplit, boxes_per_split, num_boxes, tiles_x, tiles_per_img, tap_pairs, tap_units;
};
static WgradPlan wgrad_plan(const HkConvDesc& d) {
  WgradPlan p;
  p.block_n = d.in_c % 256 == 0 ? 256 : (d.in_c % 128 == 0 ? 128 : 64);
  p.m_tiles = d.out_c <= 64 ? 1 : d.out_c / 128;
  p.n_tiles = d.in_c / p.block_n;
  p.taps = d.kh * d.kw;
  // two taps per unit (the shift on dY): the 64-output-channel convs at stride 1 with equal input / output grids, i.e. layer 1
  static const bool pairs_off = [] { const char* e = getenv("HK_WGRAD_TAP_PAIRS"); return e && e[0] == '0'; }();
  p.tap_pairs = (!pairs_off && d.out_c == 64 && d.stride == 1 && d.in_h == d.out_h && d.in_w == d.out_w && p.taps > 1) ? 1 : 0;
  p.tap_units = p.tap_pairs ? (p.taps + 1) / 2 : p.taps;
  p.tiles_x = ceil_div(d.out_w, WG_BOX_W);
  p.tiles_per_img = p.tiles_x * ceil_div(d.out_h, WG_BOX_H);
  p.num_boxes = p.tiles_per_img * d.batch;
  const int base = p.tap_units * p.m_tiles * p.n_tiles;
  // K splits: enough units for `rounds` units per persistent CTA.  One round (default since round 2): half the fp32 partials to write
  // and to reduce of the two-round plan of round 1, whose only merit -- the second unit's mainloop hiding the first one's epilogue -- is
  // matched by having half as many epilogues; batch 4: 4.07 -> 3.89 ms per step, batch 32: 22.7 -> 22.5 ms (A/B on one box).
  // HK_WGRAD_ROUNDS (read once) restores 2 for A/B runs.
  static const int rounds = [] { const char* e = getenv("HK_WGRAD_ROUNDS"); const int r = e ? atoi(e) : 0; return r >= 1 && r <= 4 ? r : 1; }();
  int ks = (rounds * sm_count()) / base;
  if (ks < 1) ks = 1;
  const int max_ks = p.num_boxes / 4 > 0 ? p.num_boxes / 4 : 1;  // at least 4 pipeline stages of work per unit
  if (ks > max_ks) ks = max_ks;
  p.boxes_per_split = ceil_div(p.num_boxes, ks);
  p.ksplit = ceil_div(p.num_boxes, p.boxes_per_split);  // every split non-empty
  return p;
}

template <int BLOCK_N>
static int launch_wgrad(const CUtensorMap& mdy, const CUtensorMap& mx, const WgradArgs& a, cudaStream_t s) {
  using Cfg = WgCfg<BLOCK_N>;
  if (int rc = opt_in_smem<conv_wgrad_kernel<BLOCK_N>>(Cfg::SMEM_BYTES, "conv wgrad")) return rc;
  const int total = a.ksplit * a.tap_units * a.m_tiles * a.n_tiles;
  int grid = sm_count();
  if (grid > total) grid = total;
  conv_wgrad_kernel<BLOCK_N><<<grid, WG_THREADS, Cfg::SMEM_BYTES, s>>>(mdy, mx, a);
  return check_launch("conv_wgrad_kernel");
}

}  // namespace hk

extern "C" {

size_t hk_conv_wgrad_workspace_bytes(const HkConvDesc* desc) {
  if (!desc || desc->in_c % 64 != 0 || desc->out_c % 64 != 0 || desc->batch <= 0) return 0;
  const hk::WgradPlan p = hk::wgrad_plan(*desc);
  return (size_t)p.ksplit * desc->out_c * p.taps * desc->in_c * sizeof(float);
}

int hk_conv_wgrad(const HkConvDesc* desc, const void* x, const void* dy, float* dw_oihw, int accumulate, void* ws, size_t ws_bytes,
                  void* stream) {
  using namespace hk;
  HK_REQUIRE(desc && x && dy && dw_oihw && ws, "hk_conv_wgrad: null pointer");
  const HkConvDesc& d = *desc;
  HK_REQUIRE(d.in_dtype == HK_BF16 && d.out_dtype == HK_BF16 && !d.in_is_nchw, "hk_conv_wgrad: needs NHWC bf16 x and dy");
  HK_REQUIRE(d.in_c % 64 == 0 && (d.out_c == 64 || d.out_c % 128 == 0), "hk_conv_wgrad: in_c %% 64 and out_c == 64 or %% 128 required (got %d, %d)",
             d.in_c, d.out_c);
  HK_REQUIRE(d.stride == 1 || d.stride == 2, "hk_conv_wgrad: stride must be 1 or 2");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(ws) & 15) == 0,
             "hk_conv_wgrad: buffers must be 16-byte aligned");
  const WgradPlan p = wgrad_plan(d);
  HK_REQUIRE(ws_bytes >= hk_conv_wgrad_workspace_bytes(desc), "hk_conv_wgrad: workspace too small");
  CUtensorMap mdy, mx;
  if (int rc = tmap_nhwc_bf16(&mdy, dy, d.batch, d.out_h, d.out_w, d.out_c, WG_BOX_W, WG_BOX_H, 1, "hk_conv_wgrad", "dy")) return rc;
  if (int rc = tmap_nhwc_bf16(&mx, x, d.batch, d.in_h, d.in_w, d.in_c, WG_BOX_W, WG_BOX_H, d.stride, "hk_conv_wgrad", "x")) return rc;
  WgradArgs a;
  a.ws = static_cast<float*>(ws);
  a.B = d.batch; a.Ho = d.out_h; a.Wo = d.out_w; a.Cout = d.out_c; a.Cin = d.in_c;
  a.kh = d.kh; a.kw = d.kw; a.stride = d.stride; a.pad = d.pad; a.dil = d.dil;
  a.tiles_x = p.tiles_x; a.tiles_per_img = p.tiles_per_img; a.num_boxes = p.num_boxes;
  a.m_tiles = p.m_tiles; a.n_tiles = p.n_tiles; a.taps = p.taps; a.ksplit = p.ksplit; a.boxes_per_split = p.boxes_per_split;
  a.cout64 = d.out_c == 64 ? 1 : 0;
  a.tap_pairs = p.tap_pairs;
  a.tap_units = p.tap_units;
  cudaStream_t s = as_stream(stream);
  int rc;
  switch (p.block_n) {
    case 256: rc = launch_wgrad<256>(mdy, mx, a, s); break;
    case 128: rc = launch_wgrad<128>(mdy, mx, a, s); break;
    default: rc = launch_wgrad<64>(mdy, mx, a, s); break;
  }
  if (rc) return rc;
  const long long total = (long long)d.out_c * p.taps * d.in_c;
  int blocks = (int)ceil_div_ll(total / 4, 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  wgrad_reduce_kernel<<<blocks, 256, 0, s>>>(a.ws, dw_oihw, p.ksplit, d.out_c, p.taps, d.in_c, accumulate);
  return check_launch("wgrad_reduce_kernel");
}

}  // extern "C"
