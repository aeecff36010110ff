// tcgen05 3x3 conv specialised for Cin = Cout = 64, stride 1 (layer1 of the backbone, reference src/resnet.py:143,
// 6 launches per forward) -- the shape whose generic implicit GEMM is bound by L2->SM operand traffic, not by the
// tensor pipe (N=64, K=576: 216 KB of operands per 128x64 output tile).
//
// Two changes against conv_tc_kernel cut that traffic 3.6x (216 KB -> 60 KB per tile):
//   * the whole weight tensor (9 taps x 64 x 64 bf16 = 72 KB) is loaded ONCE per CTA and stays in shared memory;
//   * the M tile is an 8x16 patch of output pixels, and instead of one TMA box per tap (9 per channel slice) the
//     producer loads ONE haloed box per horizontal tap s: (64 ch, 16 px, 8+2*dil rows).  In shared memory a box is
//     [row][16 px][128 B], i.e. every image row is two 1024-byte swizzle atoms, so the A operand of tap (r, s) is
//     simply the same box starting r*dil rows further down: start address + r*dil*2048, still 1024-byte aligned,
//     still the canonical K-major SWIZZLE_128B layout.  Vertical taps cost no extra loads at all.
//   * the epilogue goes through shared memory and TMA: the residual tile is TMA-loaded into a 16 KB swizzled
//     staging buffer, each epilogue thread adds its row in place, and one TMA store writes the 8x16x64 tile
//     (2 KB contiguous per image row) -- instead of 16-byte loads/stores at a 128-byte lane stride, which cost
//     8x the L1 wavefronts and made the epilogue as long as the MMA phase for this N=64 shape.
// TMEM double buffering and the warp roles follow conv_tc_kernel.
#include <cuda.h>

#include "hk_common.cuh"
#include "hk_bn_acc.cuh"
#include "hk_ptx.cuh"

namespace hk {

constexpr int C64_TILE_H = 8, C64_TILE_W = 16;   // 128 output pixels = UMMA M
constexpr int C64_C = 64;
constexpr int C64_ROW_BYTES = C64_TILE_W * 128;  // one image row of a box: 16 px x 64 ch bf16 = 2048 B
constexpr int C64_W_BYTES = 9 * C64_C * 128;     // 72 KB resident weights
constexpr int C64_THREADS = 384;   // warps 0-3: TMA producer, MMA issuer, TMEM allocator, spare; warps 4-11: epilogue
constexpr int C64_EPI_THREADS = 256;
constexpr int C64_MAX_SLOTS = 8;  // patch slots (one haloed box each); the host picks as many as fit in shared memory

struct ConvC64Args {
  const float* scale;
  const float* bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* y;
  int B, H, W, dil, relu;
  int tiles_x, tiles_per_img, num_tiles;
  int box_rows, patch_bytes;  // 8 + 2*dil rows; box_rows * 2048
  int has_residual;
  int slots;  // number of patch slots in the ring
  BnAcc* bn_acc;  // STATS kernel only: [2][64] accumulators of sum y / sum y^2 over the stored bf16 outputs (train-mode BatchNorm)
#ifdef HK_DIAG
  long long* dbg;  // optional timeline of CTA 0 (tools/diag_c64_timeline.py); diagnostics build only
#endif
};
#ifdef HK_DIAG
#define C64_STAMP(role, t, slot) \
  do { if (a.dbg && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (t) < 16) a.dbg[((role) * 16 + (t)) * 8 + (slot)] = clock64(); } while (0)
#else
#define C64_STAMP(role, t, slot) do { } while (0)
#endif
constexpr int C64_STAGING_BYTES = 128 * 128;  // one output tile: 128 pixels x 64 ch bf16 (two of them: tiles alternate)

template <bool STATS>
__global__ void __launch_bounds__(C64_THREADS, 1)
conv_tc_c64_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                   const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_res, const ConvC64Args a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sW = smem;                                    // 9 x [64 rows][128 B]
  uint8_t* sA = smem + C64_W_BYTES;                      // STAGES x 3 patches
  const int SLOTS = a.slots;
  uint8_t* sOut = sA + SLOTS * a.patch_bytes;            // epilogue staging (residual in, result out), 1024-aligned
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sOut + 2 * C64_STAGING_BYTES);
  uint64_t* empty_bar = full_bar + C64_MAX_SLOTS;
  uint64_t* tmem_full_bar = empty_bar + C64_MAX_SLOTS;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint64_t* w_bar = tmem_empty_bar + 2;
  uint64_t* res_bar = w_bar + 1;   // [2]: residual tile landed in staging buffer i
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(res_bar + 2);
  float* s_scale = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);  // [64] scale, [64] bias: broadcast reads in the epilogue
  float* s_bias = s_scale + C64_C;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp: provably uniform

  ptx::griddep_launch_dependents();  // the next kernel's CTAs may take over SMs as ours exit (its prologue overlaps our tail)
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
    ptx::prefetch_tensormap(&map_y);
    if (a.has_residual) ptx::prefetch_tensormap(&map_res);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < SLOTS; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], C64_EPI_THREADS);
    }
    ptx::mbar_init(w_bar, 1);
    ptx::mbar_init(&res_bar[0], 1);
    ptx::mbar_init(&res_bar[1], 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_ptr_smem, 128);
    ptx::tmem_relinquish();
  }
  if (warp == 3) {
    ptx::griddep_wait();  // scale / bias may have been written by the previous kernel (weight packing)
    for (int i = lane; i < C64_C; i += 32) { s_scale[i] = a.scale[i]; s_bias[i] = a.bias[i]; }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    {
      // ===================== TMA producer (whole warp waits, one elected lane issues) =====================
      ptx::griddep_wait();  // no global read (weights included) before the previous kernel has completed
      if (lane == 0) {
        ptx::mbar_arrive_expect_tx(w_bar, C64_W_BYTES);
        for (int t = 0; t < 9; ++t) ptx::tma_load_2d(sW + t * (C64_C * 128), &map_w, w_bar, t * C64_C, 0);
      }
      __syncwarp();
      uint32_t stage = 0, phase = 0;
      int dt = 0;
      for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++dt) {
        const int b = tile / a.tiles_per_img;
        const int rem = tile - b * a.tiles_per_img;
        const int ty = rem / a.tiles_x;
        const int y0 = ty * C64_TILE_H, x0 = (rem - ty * a.tiles_x) * C64_TILE_W;
        for (int s = 0; s < 3; ++s) {  // one haloed box per horizontal tap; each is its own pipeline slot
          C64_STAMP(0, dt, 2 * s);
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 21);
          C64_STAMP(0, dt, 2 * s + 1);
          if (ptx::elect_one_sync()) {
            ptx::mbar_arrive_expect_tx(&full_bar[stage], a.patch_bytes);
            ptx::tma_load_4d(sA + stage * a.patch_bytes, &map_x, &full_bar[stage], 0, x0 + (s - 1) * a.dil, y0 - a.dil, b);
          }
          __syncwarp();
          if (++stage == (uint32_t)SLOTS) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer (whole warp waits, one elected lane issues) =====================
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, C64_C);
      ptx::mbar_wait(w_bar, 0, 22);
      const uint32_t w0 = ptx::smem_u32(sW);
      uint32_t stage = 0, phase = 0, it = 0;
      for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
        C64_STAMP(1, (int)it, 0);
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, 23);
        C64_STAMP(1, (int)it, 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * C64_C;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          ptx::mbar_wait(&full_bar[stage], phase, 24);
          C64_STAMP(1, (int)it, 2 + s);
          ptx::tc_fence_after();
          const uint32_t st = ptx::smem_u32(sA + stage * a.patch_bytes);
          if (ptx::elect_one_sync()) {
#pragma unroll
            for (int r = 0; r < 3; ++r) {  // vertical taps: same box, r*dil rows further down
              const uint64_t adesc = ptx::make_smem_desc_sw128(st + r * a.dil * C64_ROW_BYTES);
              const uint64_t bdesc = ptx::make_smem_desc_sw128(w0 + (r * 3 + s) * (C64_C * 128));
#pragma unroll
              for (int k = 0; k < 4; ++k) ptx::umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (r | s | k) != 0 ? 1u : 0u);
            }
            ptx::umma_commit(&empty_bar[stage]);
            if (s == 2) ptx::umma_commit(&tmem_full_bar[acc]);
          }
          __syncwarp();
          if (++stage == (uint32_t)SLOTS) { stage = 0; phase ^= 1; }
        }
        C64_STAMP(1, (int)it, 5);
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps = 256 threads, named barrier 1) =====================
    // warp % 4 = TMEM lane quarter (32 pixels), (warp - 4) / 4 = channel half (32 of the 64 accumulator columns): the drain of one
    // tile takes half as long as with 4 warps, which were the slowest stage of the pipeline (2.4k clocks per tile against 2.0k of MMAs)
    const int q = warp & 3, half = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    ptx::griddep_wait();  // before the first residual load / output store
    const bool leader = (warp == 4 && lane == 0);
    const int sw = row & 7;
    const int et = (int)threadIdx.x - 128;   // epilogue thread 0..255
    EpiStats stats;
    if (STATS) epi_stats_init(stats, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 1024), C64_C, et);
    uint32_t it = 0;
    auto tile_origin = [&](int tile, int& b, int& y0, int& x0) {
      b = tile / a.tiles_per_img;
      const int rem = tile - b * a.tiles_per_img;
      const int ty = rem / a.tiles_x;
      y0 = ty * C64_TILE_H;
      x0 = (rem - ty * a.tiles_x) * C64_TILE_W;
    };
    // The two staging buffers alternate by tile; the residual of tile i+1 is fetched into the other buffer while tile i is
    // finished (it used to be requested at the start of its own tile: ~1.2k clocks of exposed TMA latency per tile).
    if (leader && a.has_residual && (int)blockIdx.x < a.num_tiles) {
      int b, y0, x0;
      tile_origin(blockIdx.x, b, y0, x0);
      ptx::mbar_arrive_expect_tx(&res_bar[0], C64_STAGING_BYTES);
      ptx::tma_load_4d(sOut, &map_res, &res_bar[0], 0, x0, y0, b);
    }
    for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const uint32_t buf = it & 1;
      uint8_t* stage_buf = sOut + buf * C64_STAGING_BYTES;
      uint8_t* my_row = stage_buf + row * 128;
      if (leader) C64_STAMP(2, (int)it, 0);
      if (leader) {
        ptx::bulk_wait_group_read0();  // every earlier TMA store has finished reading its staging buffer
        const int next = tile + (int)gridDim.x;
        if (a.has_residual && next < a.num_tiles) {
          int nb, ny0, nx0;
          tile_origin(next, nb, ny0, nx0);
          ptx::mbar_arrive_expect_tx(&res_bar[buf ^ 1], C64_STAGING_BYTES);
          ptx::tma_load_4d(sOut + (buf ^ 1) * C64_STAGING_BYTES, &map_res, &res_bar[buf ^ 1], 0, nx0, ny0, nb);
        }
      }
      ptx::named_bar_sync(1, C64_EPI_THREADS);  // this tile's staging buffer is free of stores (the next tile's residual is in flight)
      if (STATS) epi_stats_reduce_prev(stats, et);
      if (leader) C64_STAMP(2, (int)it, 1);
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase, 25);
      ptx::tc_fence_after();
      if (leader) C64_STAMP(2, (int)it, 2);
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * C64_C + half * 32;
      uint32_t r[32];
      ptx::tmem_ld_32x32(taddr, r);
      if (a.has_residual) ptx::mbar_wait(&res_bar[buf], (it >> 1) & 1, 26);
      if (leader) C64_STAMP(2, (int)it, 3);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&tmem_empty_bar[acc]);  // accumulator drained into registers: the MMA warp may start tile it+2
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int c = half * 32 + g * 8;
        const float4 s0 = *reinterpret_cast<const float4*>(s_scale + c);
        const float4 s1 = *reinterpret_cast<const float4*>(s_scale + c + 4);
        const float4 t0 = *reinterpret_cast<const float4*>(s_bias + c);
        const float4 t1 = *reinterpret_cast<const float4*>(s_bias + c + 4);
        const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float bi[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(__uint_as_float(r[g * 8 + j]), sc[j], bi[j]);
        uint4* slot = reinterpret_cast<uint4*>(my_row + ((((c >> 3) ^ sw) & 7) << 4));  // 128-byte swizzle, as TMA expects
        if (a.has_residual) {
          const uint4 rr = *slot;
          float lo, hi;
          unpack_bf16x2(rr.x, lo, hi); v[0] += lo; v[1] += hi;
          unpack_bf16x2(rr.y, lo, hi); v[2] += lo; v[3] += hi;
          unpack_bf16x2(rr.z, lo, hi); v[4] += lo; v[5] += hi;
          unpack_bf16x2(rr.w, lo, hi); v[6] += lo; v[7] += hi;
        }
        if (a.relu) {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        *slot = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      }
      if (leader) C64_STAMP(2, (int)it, 4);
      ptx::fence_proxy_async_smem();           // my smem writes -> visible to the TMA store
      ptx::named_bar_sync(1, C64_EPI_THREADS);
      if (leader) C64_STAMP(2, (int)it, 5);
      if (leader) {
        int b, y0, x0;
        tile_origin(tile, b, y0, x0);
        ptx::tma_store_4d(&map_y, stage_buf, 0, x0, y0, b);  // rows / columns beyond the image are clipped
        ptx::bulk_commit_group();
      }
      if (STATS) {   // this thread's 16 staged rows = 16 pixels of image row y0 + (et >> 5)
        int b, y0, x0;
        tile_origin(tile, b, y0, x0);
        const int nvalid = (y0 + (et >> 5) < a.H) ? min(16, max(0, a.W - x0)) : 0;
        epi_stats_chunk(stats, stage_buf, et, nvalid, 0);
      }
    }
    if (STATS) epi_stats_flush(stats, et, C64_C, a.bn_acc, [] { ptx::named_bar_sync(1, C64_EPI_THREADS); });
    if (leader) ptx::bulk_wait_group0();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 128);
  }
}

#ifdef HK_DIAG
static long long* g_c64_dbg = nullptr;
extern "C" __attribute__((visibility("default"))) void hk_debug_set_c64_timeline(long long* dev_buf) { g_c64_dbg = dev_buf; }
#endif

bool conv_tc_c64_applicable(const HkConvDesc& d) {
  if (!(d.kh == 3 && d.kw == 3 && d.stride == 1 && d.in_c == 64 && d.out_c == 64 && d.pad == d.dil)) return false;
  const int box_rows = C64_TILE_H + 2 * d.dil;
  const int smem_min = 1024 + C64_W_BYTES + 3 * box_rows * C64_ROW_BYTES + 2 * C64_STAGING_BYTES + 1024;  // at least one tile in flight
  return box_rows <= 256 && smem_min <= 227 * 1024;
}

int conv_tc_c64_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                       const void* residual, void* y, void* bn_acc, cudaStream_t s) {
  const int box_rows = C64_TILE_H + 2 * d.dil;
  const char* who = "conv(tcgen05,c64)";
  CUtensorMap mx, mw, my, mres;
  if (int rc = tmap_nhwc_bf16(&mx, x, d.batch, d.in_h, d.in_w, d.in_c, C64_TILE_W, box_rows, 1, who, "activations")) return rc;
  if (int rc = tmap_kmajor_bf16(&mw, w, 9 * 64, 64, 64, who, "weights")) return rc;
  if (int rc = tmap_nhwc_bf16(&my, y, d.batch, d.out_h, d.out_w, 64, C64_TILE_W, C64_TILE_H, 1, who, "output")) return rc;
  mres = my;
  if (residual) {
    if (int rc = tmap_nhwc_bf16(&mres, residual, d.batch, d.out_h, d.out_w, 64, C64_TILE_W, C64_TILE_H, 1, who, "residual")) return rc;
  }
  ConvC64Args a;
  a.has_residual = residual ? 1 : 0;
#ifdef HK_DIAG
  a.dbg = g_c64_dbg;
#endif
  a.scale = scale; a.bias = bias;
  a.residual = static_cast<const __nv_bfloat16*>(residual);
  a.y = static_cast<__nv_bfloat16*>(y);
  a.B = d.batch; a.H = d.out_h; a.W = d.out_w; a.dil = d.dil; a.relu = d.relu;
  a.tiles_x = ceil_div(d.out_w, C64_TILE_W);
  a.tiles_per_img = a.tiles_x * ceil_div(d.out_h, C64_TILE_H);
  const long long nt = (long long)a.tiles_per_img * d.batch;
  HK_REQUIRE(nt < 0x7fffffffLL, "conv(tcgen05,c64): too many tiles");
  a.num_tiles = (int)nt;
  a.box_rows = box_rows;
  a.patch_bytes = box_rows * C64_ROW_BYTES;
  a.bn_acc = static_cast<BnAcc*>(bn_acc);
  // alignment slack, weights, staging, barriers + scale/bias (1 KB), the epilogue's statistics scratch (STATS kernel)
  const int fixed = 1024 + C64_W_BYTES + 2 * C64_STAGING_BYTES + 1024 + (bn_acc ? epi_stats_smem_bytes(C64_C) : 0);
  int slots = (227 * 1024 - fixed) / a.patch_bytes;
  if (slots > C64_MAX_SLOTS) slots = C64_MAX_SLOTS;
  a.slots = slots;
  const int smem = fixed + slots * a.patch_bytes;
  if (int rc = bn_acc ? opt_in_smem<conv_tc_c64_kernel<true>>(smem, who) : opt_in_smem<conv_tc_c64_kernel<false>>(smem, who)) return rc;
  int grid = sm_count();
  if (grid > a.num_tiles) grid = a.num_tiles;
  cudaError_t le = bn_acc ? launch_pdl(conv_tc_c64_kernel<true>, dim3(grid), dim3(C64_THREADS), (size_t)smem, s, mx, mw, my, mres, a)
                          : launch_pdl(conv_tc_c64_kernel<false>, dim3(grid), dim3(C64_THREADS), (size_t)smem, s, mx, mw, my, mres, a);
  if (le != cudaSuccess) return fail(HK_ERR_CUDA, "conv_tc_c64_kernel: %s", cudaGetErrorString(le));
  return check_launch("conv_tc_c64_kernel");
}

}  // namespace hk
