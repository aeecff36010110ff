// Fused stem for inference: conv 7x7 stride 2 pad 3 (3 -> 64) + folded BN + ReLU + MaxPool2d(3, 2, 1) in ONE kernel,
// bf16 operands / fp32 accumulate on tcgen05, pooled bf16 NHWC out.
//
// Replaces nn.Conv2d(3,64,7,2,3) -> BatchNorm2d(eval) -> ReLU -> MaxPool2d(3,2,1) of reference src/resnet.py:137-141,199-202.
// The two-kernel path (stem_tc_kernel + maxpool3x3s2_kernel) writes the (B,H/2,W/2,64) stem map to HBM and reads it back
// (629 MB + 629 MB at batch 64) and spends most of its time copying im2col rows through shared memory.  Here neither happens:
//
//  * Row streaming.  A CTA owns a strip of 128 stem columns and walks it top to bottom, one stem row (= one M=128 MMA tile)
//    at a time.  A stem row needs input rows 2y-3 .. 2y+3: the input lives in a shared-memory ring of 16 rows, two new rows per
//    step arrive by TMA (fp32 NCHW planes or uint8 HWC rows; out-of-image elements are zero-filled by the TMA unit = the
//    conv's padding) and are rounded to bf16 as [x][4] (three channels + a zero: one pixel = 8 bytes) by four converter warps.
//  * No im2col copy.  With 8-byte pixels and stride 2, consecutive stem outputs of one row are exactly 16 bytes apart in the
//    ring, and the 7 taps x 3 channels of filter row r are 64 contiguous bytes.  That IS a K-major UMMA operand in the
//    no-swizzle ("interleave") canonical layout ((8,m),(8,2)):((16 B, SBO = 128 B),(2 B, LBO = 16 B)): core matrices overlap
//    (row i, 16-byte K chunk j sits at byte 16*(i+j)), which a read-only operand may.  The A descriptor of filter row r just
//    points at ring row 2y-3+r; 14 tcgen05.mma (M=128, N=64, K=16) per stem row against the SWIZZLE_128B weights.
//  * Pooling in registers.  Each epilogue thread owns one stem column x 32 channels: it keeps the running vertical maximum of
//    relu(scale*acc+bias) in fp32 registers (max commutes with the monotone bf16 rounding, so the result is bit-identical to
//    pooling the rounded stem map); every second row the 128-column row of maxima goes through a swizzled shared buffer for the
//    horizontal 3-max and leaves as 16-byte coalesced stores of pooled bf16 NHWC.
//    Strips overlap by two stem columns (126 useful of 128: the window of pooled column j is stem columns 2j-1 .. 2j+1), bands
//    of rows recompute one carry row: 3 % extra MMA work instead of the 33 % of a 9x17 tile.
//
// Warp roles (512 threads, 1 CTA/SM): 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4-7 = converters, 8-15 = epilogue.
#include <cuda.h>
#include <stdlib.h>

#include "hk_common.cuh"
#include "hk_ptx.cuh"

namespace hk {

constexpr int SP_THREADS = 512;
constexpr int SP_USE = 126;                     // useful stem columns per strip -> 63 pooled columns
constexpr int SP_POOL = 63;
constexpr int SP_PX = 264;                      // input pixels per ring row: 2*127 + 7 + 1 = 262, padded
constexpr int SP_ROW_BYTES = SP_PX * 8;         // 2112
constexpr int SP_PAIR_BYTES = 2 * SP_ROW_BYTES; // a ring slot holds an even/odd input row pair
constexpr int SP_PAIRS = 8;
constexpr int SP_RING_BYTES = SP_PAIRS * SP_PAIR_BYTES;      // 33792
constexpr int SP_STAGES = 4;
constexpr int SP_ACC = 2;                       // TMEM accumulators (64 columns each); 4 (the epilogue three rows behind the MMAs) measured no faster
// TMA needs the box to START on a 16-byte boundary in global memory (an unaligned innermost coordinate raises an illegal-instruction
// fault): the fp32 box starts 3 pixels left of ring pixel 0 (input column 252*strip - 8, a multiple of 4 floats), the uint8 box at the
// 16-byte boundary below byte 3*(252*strip - 5); the converters skip the lead-in.
constexpr int SP_F32_LEAD = 3;
constexpr int SP_F32_BOX = 136;                 // fp32: two boxes of 136 columns x 2 rows x 3 planes per pair (TMA boxes are <= 256 wide)
constexpr int SP_F32_BOX_BYTES = 3 * 2 * SP_F32_BOX * 4;     // 3264 bytes land per box ...
constexpr int SP_F32_BOX_PITCH = 3328;          // ... at 128-byte aligned addresses (TMA destination alignment)
constexpr int SP_F32_TX = 2 * SP_F32_BOX_BYTES;
constexpr int SP_U8_BOX = 208;                  // uint8: four boxes of 208 bytes x 2 rows per pair (792 bytes + up to 15 of lead-in needed)
constexpr int SP_U8_BOX_BYTES = 2 * SP_U8_BOX;  // 416
constexpr int SP_U8_BOX_PITCH = 512;
constexpr int SP_U8_TX = 4 * SP_U8_BOX_BYTES;
constexpr int SP_STAGE_BYTES = 2 * SP_F32_BOX_PITCH;         // 6656; both instantiations use the larger size
constexpr int SP_B_BYTES = 64 * 128 * 4;        // weights: 4 K blocks x [64 rows][128 B], SWIZZLE_128B
constexpr int SP_P_BYTES = 128 * 128;           // one row of vertical maxima: 128 columns x 64 ch bf16 (two buffers)
constexpr int SP_EPI_THREADS = 256;
constexpr int SP_CONV_THREADS = 128;
constexpr int SP_SMEM_BYTES = 1024 + SP_B_BYTES + SP_RING_BYTES + SP_STAGES * SP_STAGE_BYTES + 2 * SP_P_BYTES + 512 + 2 * 64 * 4;

struct StemPoolArgs {
  const float* scale;
  const float* bias;
  __nv_bfloat16* y;  // (B,Hp,Wp,64) bf16 pooled
  int B, H, W, Ho, Wo, Hp, Wp;
  int band_rows;     // stem rows per band (even)
  int nbands, nstrips, num_units;
#ifdef HK_DIAG
  int dbg_mode;   // HK_SP_DEBUG bit flags (diagnostics build): 1 = no TMA input loads, 2 = no MMAs, 4 = no epilogue TMEM loads,
                  // 8 = converters only pass their barriers on, 16 = epilogue stops after releasing the accumulator
#endif
};
#ifdef HK_DIAG
#define SP_DBG(a) ((a).dbg_mode)
#else
#define SP_DBG(a) 0
#endif

// K-major operand, no swizzle: 8-row core matrices of 16-byte rows; LBO = byte distance of the two K chunks of one MMA,
// SBO = byte distance of consecutive 8-row groups.
__device__ __forceinline__ uint64_t make_smem_desc_nosw(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(ptx::smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(ptx::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// first byte of the uint8 TMA box: the 16-byte boundary at or below byte 3*x_start of the row (x_start may be negative)
__device__ __forceinline__ int sp_u8_aligned_start(int x_start) {
  const int b0 = 3 * x_start;
  return b0 - (((b0 % 16) + 16) % 16);
}

struct SpUnit {
  int b, strip, y_first, y_end, y0;  // stem rows [y_first, y_end); y0 = first row of the band (y_first = y0 - 1 when a carry row is needed)
  int rows;                          // y_end - y_first
};
__device__ __forceinline__ SpUnit sp_unit(const StemPoolArgs& a, int u) {
  SpUnit r;
  r.strip = u % a.nstrips;
  const int t = u / a.nstrips;
  const int band = t % a.nbands;
  r.b = t / a.nbands;
  r.y0 = band * a.band_rows;
  r.y_first = r.y0 > 0 ? r.y0 - 1 : 0;
  r.y_end = min(r.y0 + a.band_rows, a.Ho);
  r.rows = r.y_end - r.y_first;
  return r;
}

template <bool U8>
__global__ void __launch_bounds__(SP_THREADS, 1)
stem_pool_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const StemPoolArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sB = smem;                               // 4 x [64][128 B] swizzled
  uint8_t* ring = sB + SP_B_BYTES;                  // 8 pairs x 2 rows x [264 px][4] bf16
  uint8_t* stages = ring + SP_RING_BYTES;           // 4 x TMA landing zone of one input row pair
  uint8_t* sP = stages + SP_STAGES * SP_STAGE_BYTES;  // 2 x [128 columns][128 B] (16-byte chunks XOR-swizzled by column & 7)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * SP_P_BYTES);
  uint64_t* stage_full = bars;                      // [4]
  uint64_t* stage_empty = bars + 4;                 // [4]
  uint64_t* pair_full = bars + 8;                   // [8]
  uint64_t* pair_empty = bars + 16;                 // [8]
  uint64_t* tmem_full = bars + 24;                  // [SP_ACC]
  uint64_t* tmem_empty = bars + 28;                 // [SP_ACC]
  uint64_t* w_bar = bars + 32;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 34);
  float* s_scale = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 512);
  float* s_bias = s_scale + 64;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

  if (tid == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
    for (int i = 0; i < SP_STAGES; ++i) {
      ptx::mbar_init(&stage_full[i], 1);
      ptx::mbar_init(&stage_empty[i], SP_CONV_THREADS);
    }
    for (int i = 0; i < SP_PAIRS; ++i) {
      ptx::mbar_init(&pair_full[i], SP_CONV_THREADS);
      ptx::mbar_init(&pair_empty[i], 1);
    }
    for (int i = 0; i < SP_ACC; ++i) {
      ptx::mbar_init(&tmem_full[i], 1);
      ptx::mbar_init(&tmem_empty[i], SP_EPI_THREADS);
    }
    ptx::mbar_init(w_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_ptr_smem, SP_ACC * 64);
    ptx::tmem_relinquish();
  }
  if (tid >= 64 && tid < 128) {
    s_scale[tid - 64] = a.scale[tid - 64];
    s_bias[tid - 64] = a.bias[tid - 64];
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer: weights once, then one input row pair per stage =====================
    if (ptx::elect_one_sync()) {
      ptx::mbar_arrive_expect_tx(w_bar, SP_B_BYTES);
      for (int kb = 0; kb < 4; ++kb) ptx::tma_load_2d(sB + kb * 8192, &map_w, w_bar, kb * 64, 0);
    }
    __syncwarp();
    uint32_t n = 0;  // running pair counter
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const SpUnit un = sp_unit(a, u);
      const int x_start = 2 * (SP_USE * un.strip - 1) - 3;     // input column of ring pixel 0
      const int q0 = un.y_first - 2;                             // first input row pair (rows 2q, 2q+1)
      const int npairs = un.rows + 3;
      for (int j = 0; j < npairs; ++j, ++n) {
        const uint32_t st = n & (SP_STAGES - 1);
        ptx::mbar_wait(&stage_empty[st], ((n >> 2) & 1) ^ 1, 41);
        if (ptx::elect_one_sync()) {
          uint8_t* dst = stages + st * SP_STAGE_BYTES;
          const int row = 2 * (q0 + j);
          if (SP_DBG(a) & 1) {
            ptx::mbar_arrive(&stage_full[st]);
          } else if constexpr (U8) {
            ptx::mbar_arrive_expect_tx(&stage_full[st], SP_U8_TX);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              tma_load_3d(dst + k * SP_U8_BOX_PITCH, &map_x, &stage_full[st], sp_u8_aligned_start(x_start) + k * SP_U8_BOX, row, un.b);
          } else {
            ptx::mbar_arrive_expect_tx(&stage_full[st], SP_F32_TX);
#pragma unroll
            for (int k = 0; k < 2; ++k)
              ptx::tma_load_4d(dst + k * SP_F32_BOX_PITCH, &map_x, &stage_full[st], x_start - SP_F32_LEAD + k * SP_F32_BOX, row, 0, un.b);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, 64);
    ptx::mbar_wait(w_bar, 0, 42);
    const uint32_t b0 = ptx::smem_u32(sB), ring0 = ptx::smem_u32(ring);
    uint32_t n0 = 0, it = 0;   // n0: pair counter at the start of the unit; it: stem rows issued so far (accumulator select)
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const SpUnit un = sp_unit(a, u);
      // pairs 0..2 of the unit must have landed before the first row; afterwards one new pair per row
      for (int j = 0; j < 3; ++j) ptx::mbar_wait(&pair_full[(n0 + j) & 7], ((n0 + j) >> 3) & 1, 43);
      for (int t = 0; t < un.rows; ++t, ++it) {
        const uint32_t acc = it & (SP_ACC - 1), acc_phase = (it / SP_ACC) & 1;
        ptx::mbar_wait(&pair_full[(n0 + t + 3) & 7], ((n0 + t + 3) >> 3) & 1, 44);
        ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1, 45);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 64;
        if (ptx::elect_one_sync()) {
#pragma unroll
          for (int r = 0; r < 7; ++r) {
            // filter row r reads input row 2y-3+r: local pair t + (r+1)/2, second row of the pair when r is even
            const uint32_t slot = (n0 + t + ((r + 1) >> 1)) & 7;
            const uint32_t arow = ring0 + slot * SP_PAIR_BYTES + ((r & 1) ? 0 : SP_ROW_BYTES);
            const uint64_t bdesc = ptx::make_smem_desc_sw128(b0 + (r >> 1) * 8192) + ((r & 1) * 4);
#pragma unroll
            for (int h = 0; h < 2; ++h)
              if (!(SP_DBG(a) & 2)) ptx::umma_bf16(d_tmem, make_smem_desc_nosw(arow + 32 * h, 16, 128), bdesc + 2 * h, idesc, (r | h) != 0 ? 1u : 0u);
          }
          ptx::umma_commit(&pair_empty[(n0 + t) & 7]);        // the oldest pair of this row is not needed by any later row
          if (t == un.rows - 1) {                             // end of the unit: release its last three pairs as well
            ptx::umma_commit(&pair_empty[(n0 + t + 1) & 7]);
            ptx::umma_commit(&pair_empty[(n0 + t + 2) & 7]);
            ptx::umma_commit(&pair_empty[(n0 + t + 3) & 7]);
          }
          ptx::umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
      }
      n0 += un.rows + 3;
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== converters: TMA landing zone -> bf16 [x][4] ring rows =====================
    const int ct = tid - 128;
    uint32_t n = 0;
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const SpUnit un = sp_unit(a, u);
      const int npairs = un.rows + 3;
      const int x_start = 2 * (SP_USE * un.strip - 1) - 3;
      const int u8_lead = 3 * x_start - sp_u8_aligned_start(x_start);   // bytes between the aligned box start and ring pixel 0
      (void)u8_lead;
      for (int j = 0; j < npairs; ++j, ++n) {
        const uint32_t st = n & (SP_STAGES - 1), slot = n & 7;
        ptx::mbar_wait(&stage_full[st], (n >> 2) & 1, 46);
        ptx::mbar_wait(&pair_empty[slot], ((n >> 3) & 1) ^ 1, 47);
        const uint8_t* src = stages + st * SP_STAGE_BYTES;
        uint8_t* dst = ring + slot * SP_PAIR_BYTES;
        if (SP_DBG(a) & 8) {
          ptx::mbar_arrive(&pair_full[slot]);
          ptx::mbar_arrive(&stage_empty[st]);
          continue;
        }
#pragma unroll
        for (int i = 0; i < (2 * SP_PX + SP_CONV_THREADS - 1) / SP_CONV_THREADS; ++i) {
          const int p = ct + i * SP_CONV_THREADS;
          if (p < 2 * SP_PX) {
            const int row = p >= SP_PX ? 1 : 0, x = p - row * SP_PX;
            float f0, f1, f2;
            if constexpr (U8) {
              // byte 3x+c of the row lives in box (3x+c)/208; ToTensor semantics (reference dataset.py:16): bf16_rn(uint8 / 255) == bf16_rn(uint8 * kInv255), see hk_common.cuh
              const int e = 3 * x + u8_lead;
              auto at = [&](int byte) { const int k = byte / SP_U8_BOX; return src[k * SP_U8_BOX_PITCH + row * SP_U8_BOX + (byte - k * SP_U8_BOX)]; };
              f0 = (float)at(e) * kInv255;
              f1 = (float)at(e + 1) * kInv255;
              f2 = (float)at(e + 2) * kInv255;
            } else {
              const int xs = x + SP_F32_LEAD;
              const int k = xs >= SP_F32_BOX ? 1 : 0, xi = xs - k * SP_F32_BOX;
              const float* s = reinterpret_cast<const float*>(src + k * SP_F32_BOX_PITCH) + row * SP_F32_BOX + xi;  // [plane][row][132]
              f0 = s[0];
              f1 = s[2 * SP_F32_BOX];
              f2 = s[4 * SP_F32_BOX];
            }
            *reinterpret_cast<uint2*>(dst + row * SP_ROW_BYTES + x * 8) = make_uint2(pack_bf16x2(f0, f1), pack_bf16x2(f2, 0.f));
          }
        }
        ptx::fence_proxy_async_smem();          // ring rows are read by tcgen05 (async proxy)
        ptx::mbar_arrive(&pair_full[slot]);
        ptx::mbar_arrive(&stage_empty[st]);
      }
    }
  } else if (warp >= 8) {
    // ===================== epilogue: affine + ReLU + 3x3/2 max pooling =====================
    const int q = warp & 3, half = (warp - 8) >> 2;
    const int col = q * 32 + lane;             // column of the strip = TMEM lane
    const int et = tid - 256;
    const int c0 = half * 32;
    // Pooling on the RAW accumulators: relu(scale*a + bias) is monotone in a (non-decreasing for scale >= 0, non-increasing for scale < 0)
    // and so is the bf16 rounding, so the maximum over a pooling window of the activated values is the activation of the window's largest
    // (smallest, for a negative scale) accumulator -- bit for bit.  The per-row work is two FMNMX per channel; affine + ReLU + bf16 pack and
    // the scale/bias reads happen once per POOLED row.  (Applying them to every stem row cost ~350 instructions per thread and row and made
    // this role the kernel's bound: 0.23 of its 0.31 ms, tools/diag_stem_pool_modes.py.)
    float amax[32], amin[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) { amax[j] = -INFINITY; amin[j] = INFINITY; }
    uint32_t it = 0, emits = 0;
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const SpUnit un = sp_unit(a, u);
      const int stem_col = SP_USE * un.strip - 1 + col;
      const bool col_ok = stem_col >= 0 && stem_col < a.Wo;
      const int px0 = SP_POOL * un.strip;      // first pooled column of the strip
      for (int t = 0; t < un.rows; ++t, ++it) {
        const uint32_t acc = it & (SP_ACC - 1), acc_phase = (it / SP_ACC) & 1;
        const int y = un.y_first + t;
        ptx::mbar_wait(&tmem_full[acc], acc_phase, 48);
        ptx::tc_fence_after();
        uint32_t r[32];
        if (SP_DBG(a) & 4) {
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = 0;
        } else {
          ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * 64 + c0, r);
          ptx::tmem_ld_wait();
        }
        ptx::tc_fence_before();
        ptx::mbar_arrive(&tmem_empty[acc]);
        if (SP_DBG(a) & 16) continue;
        const bool carry_only = (t == 0 && un.y0 > 0);          // row y0-1: the first row of the band's first pooling window
        const bool emit = !carry_only && ((y & 1) || y == a.Ho - 1);
        if (carry_only || t == 0) {   // first row of a window sequence (band 0 has no row above)
#pragma unroll
          for (int j = 0; j < 32; ++j) { amax[j] = __uint_as_float(r[j]); amin[j] = __uint_as_float(r[j]); }
          if (carry_only) continue;
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            amax[j] = fmaxf(amax[j], __uint_as_float(r[j]));
            amin[j] = fminf(amin[j], __uint_as_float(r[j]));
          }
        }
        if (!emit) continue;
        // ---- pooled row py = y >> 1: activation of the window extremes -> swizzled smem row, horizontal 3-max, coalesced 16-byte stores ----
        uint8_t* P = sP + (emits & 1) * SP_P_BYTES;
        ++emits;
        {
          uint8_t* my = P + col * 128;
          const int sw = col & 7;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int cc = half * 4 + i;
            float v[8];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              const float4 s4 = *reinterpret_cast<const float4*>(s_scale + c0 + i * 8 + g * 4);
              const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c0 + i * 8 + g * 4);
              const float sc[4] = {s4.x, s4.y, s4.z, s4.w}, bi[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = i * 8 + g * 4 + e;
                const float ext = sc[e] >= 0.f ? amax[j] : amin[j];
                // outside the stem map: MaxPool's padding never wins (activated values are >= 0)
                v[g * 4 + e] = col_ok ? fmaxf(fmaf(ext, sc[e], bi[e]), 0.f) : 0.f;
              }
            }
            *reinterpret_cast<uint4*>(my + ((cc ^ sw) << 4)) =
                make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          }
        }
        // the next window starts with this row when it is odd (row 2py+1 = row 2(py+1)-1)
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          amax[j] = (y & 1) ? __uint_as_float(r[j]) : -INFINITY;
          amin[j] = (y & 1) ? __uint_as_float(r[j]) : INFINITY;
        }
        ptx::named_bar_sync(1, SP_EPI_THREADS);
        const int py = y >> 1;
        __nv_bfloat16* out_row = a.y + ((size_t)(un.b * a.Hp + py) * a.Wp) * 64;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int idx = et + i * SP_EPI_THREADS;      // 63 pooled columns x 8 chunks of 16 bytes
          const int j = idx >> 3, cc = idx & 7;
          if (j < SP_POOL && px0 + j < a.Wp) {
            const uint4 p0 = *reinterpret_cast<const uint4*>(P + (2 * j) * 128 + ((cc ^ ((2 * j) & 7)) << 4));
            const uint4 p1 = *reinterpret_cast<const uint4*>(P + (2 * j + 1) * 128 + ((cc ^ ((2 * j + 1) & 7)) << 4));
            const uint4 p2 = *reinterpret_cast<const uint4*>(P + (2 * j + 2) * 128 + ((cc ^ ((2 * j + 2) & 7)) << 4));
            auto mx = [](uint32_t x, uint32_t y2, uint32_t z) {
              __nv_bfloat162 m = __hmax2(__hmax2(*reinterpret_cast<__nv_bfloat162*>(&x), *reinterpret_cast<__nv_bfloat162*>(&y2)),
                                         *reinterpret_cast<__nv_bfloat162*>(&z));
              return *reinterpret_cast<uint32_t*>(&m);
            };
            const uint4 o = make_uint4(mx(p0.x, p1.x, p2.x), mx(p0.y, p1.y, p2.y), mx(p0.z, p1.z, p2.z), mx(p0.w, p1.w, p2.w));
            *reinterpret_cast<uint4*>(out_row + (size_t)(px0 + j) * 64 + cc * 8) = o;
          }
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, SP_ACC * 64);
  }
}

static int stem_pool_launch(const void* x, bool u8, const void* w_packed, const float* scale, const float* bias, void* y, int B, int H,
                            int W, void* stream) {
  HK_REQUIRE(x && w_packed && scale && bias && y, "hk_stem_pool_fwd: null pointer");
  HK_REQUIRE(B > 0 && H >= 7 && W >= 7, "hk_stem_pool_fwd: bad shape");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(w_packed) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(x) & 15) == 0, "hk_stem_pool_fwd: buffers must be 16-byte aligned");
  // TMA row pitch must be a multiple of 16 bytes
  HK_REQUIRE(u8 ? (3 * W) % 16 == 0 : W % 4 == 0, "hk_stem_pool_fwd: W must be a multiple of %d for the TMA input path", u8 ? 16 : 4);
  const char* who = "hk_stem_pool_fwd";
  CUtensorMap mw, mx;
  if (int rc = tmap_kmajor_bf16(&mw, w_packed, 256, 64, 64, who, "weights")) return rc;
  if (u8) {
    const cuuint64_t dims[3] = {(cuuint64_t)3 * W, (cuuint64_t)H, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)3 * W, (cuuint64_t)3 * W * H};
    const cuuint32_t box[3] = {(cuuint32_t)SP_U8_BOX, 2, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    if (int rc = tmap_encode(&mx, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, x, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, who, "uint8 input"))
      return rc;
  } else {
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, 3, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4, (cuuint64_t)W * H * 12};
    const cuuint32_t box[4] = {(cuuint32_t)SP_F32_BOX, 2, 3, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (int rc = tmap_encode(&mx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, x, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, who, "fp32 input"))
      return rc;
  }
  StemPoolArgs a;
  a.scale = scale; a.bias = bias; a.y = static_cast<__nv_bfloat16*>(y);
  a.B = B; a.H = H; a.W = W;
  a.Ho = (H + 6 - 7) / 2 + 1;
  a.Wo = (W + 6 - 7) / 2 + 1;
  a.Hp = (a.Ho + 2 - 3) / 2 + 1;
  a.Wp = (a.Wo + 2 - 3) / 2 + 1;
  a.nstrips = ceil_div(a.Wp, SP_POOL);
  // bands of stem rows: each band recomputes one carry row, so prefer few bands -- but enough units to balance the persistent grid
  int band = 40;
  const int sms = sm_count();
  while (band > 8 && (long long)B * a.nstrips * ceil_div(a.Ho, band) < 4LL * sms) band -= 8;
  a.band_rows = band;
  a.nbands = ceil_div(a.Ho, band);
  const long long units = (long long)B * a.nbands * a.nstrips;
  HK_REQUIRE(units < 0x7fffffffLL, "hk_stem_pool_fwd: too many work units");
  a.num_units = (int)units;
#ifdef HK_DIAG
  { const char* m = getenv("HK_SP_DEBUG"); a.dbg_mode = m ? atoi(m) : 0; }
#endif
  if (int rc = u8 ? opt_in_smem<stem_pool_kernel<true>>(SP_SMEM_BYTES, who) : opt_in_smem<stem_pool_kernel<false>>(SP_SMEM_BYTES, who)) return rc;
  int grid = sms;
  if (grid > a.num_units) grid = a.num_units;
  if (u8) stem_pool_kernel<true><<<grid, SP_THREADS, SP_SMEM_BYTES, as_stream(stream)>>>(mx, mw, a);
  else stem_pool_kernel<false><<<grid, SP_THREADS, SP_SMEM_BYTES, as_stream(stream)>>>(mx, mw, a);
  return check_launch("stem_pool_kernel");
}

}  // namespace hk

extern "C" {

#ifdef HK_DIAG
// diagnostics build: (site, block, thread, parity) of the first stuck mbarrier wait of this translation unit's kernels; clears it
__attribute__((visibility("default"))) int hk_debug_read_watchdog_stem_pool(unsigned int* out4) {
  cudaError_t e = cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out4, hk::ptx::hk_watchdog, 16);
  unsigned int zero[4] = {0, 0, 0, 0};
  cudaMemcpyToSymbol(hk::ptx::hk_watchdog, zero, 16);
  cudaMemcpyToSymbol(hk::ptx::hk_watchdog_abort, zero, 4);
  return (int)e;
}
#endif

int hk_stem_pool_fwd(const float* x_nchw, const void* w_packed, const float* scale, const float* bias, void* y_pooled_nhwc, int B,
                     int H, int W, void* stream) {
  return hk::stem_pool_launch(x_nchw, false, w_packed, scale, bias, y_pooled_nhwc, B, H, W, stream);
}

int hk_stem_pool_fwd_u8(const uint8_t* x_nhwc_u8, const void* w_packed, const float* scale, const float* bias, void* y_pooled_nhwc,
                        int B, int H, int W, void* stream) {
  return hk::stem_pool_launch(x_nhwc_u8, true, w_packed, scale, bias, y_pooled_nhwc, B, H, W, stream);
}

}  // extern "C"
