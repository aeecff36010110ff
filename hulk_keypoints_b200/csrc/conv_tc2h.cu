// Haloed-operand variant of the 2-CTA tcgen05 convolution (conv_tc2.cu) for 3x3 stride-1 convs whose mainloop is bound by
// L2->SM operand traffic (the 128-channel layer: 24 KB per K block per CTA at ~12 TB/s chip-wide, MMAs idle half the time).
//
// Same math and protocol as conv_tc2_kernel; what changes is how the activation operand reaches shared memory:
//   * each CTA's 128 accumulator rows are ONE 8x16 patch of output pixels (the pair covers two patches) instead of two 4x16 boxes;
//   * per horizontal tap s and 64-channel block the producer loads ONE box (64 ch, 16 px, 8 + 2*dil rows) at x0 + (s-1)*dil, y0 - dil.
//     With SWIZZLE_128B it lands as [(8+2*dil)*16 pixels][128 B]; the A operand of vertical tap r is the same tile r*dil rows
//     (= r*dil*2048 bytes, still 1024-byte aligned, still the canonical K-major layout) further down -- the three vertical taps cost
//     one load: 20 / 24 / 32 KB (dil 1 / 2 / 4) instead of 3 x 16 KB;
//   * weights stream through their own ring, one (tap, channel block) tile per stage, half of the BLOCK_N rows per CTA as before.
// Two rings (A: haloed boxes, B: weight tiles), each with full (leader's smem, 2 arrivals + both CTAs' TMA bytes) / empty (both
// CTAs, multicast commit) barriers; accumulate order is (s, channel block, r).  Epilogue as in conv_tc2 with one 8x16 box per chunk.
// A feature map whose height is 1..4 rows past a multiple of 8 (60 = 7 x 8 + 4) would waste half of its last 8-row patch row (6.7 % of
// the MMAs at 60 rows): those bottom rows are covered by 4x32 STRIP patches instead -- same 128 accumulator rows, box (64 ch, 32 px,
// 4 + 2*dil rows), vertical taps r*dil*4096 bytes apart.  Full patches are enumerated first, strips after them, and the boundary is
// padded to an even index, because both CTAs of a pair must work on the same patch shape (the tap offset is part of the ONE A
// descriptor of the cta_group::2 MMA).
#include <cuda.h>

#include "hk_common.cuh"
#include "hk_bn_acc.cuh"
#include "hk_ptx.cuh"
#include "hk_ptx2.cuh"

namespace hk {

constexpr int TH_TILE_H = 8, TH_TILE_W = 16;
constexpr int TH_ROW_BYTES = TH_TILE_W * 128;  // one patch row: 16 px x 64 ch bf16
constexpr int TH_THREADS = 384;   // warps 0-3: TMA producer, MMA issuer, TMEM allocator, spare; warps 4-11: epilogue
constexpr int TH_EPI_THREADS = 256;
constexpr int TH_STAGING_BYTES = 3 * 128 * 128;
constexpr int TH_MAX_A = 4, TH_MAX_B = 8;

struct ConvTc2hArgs {
  const float* scale;
  const float* bias;
  const __nv_bfloat16* residual;
  int B, Ho, Wo, Cout, Cin, pad, dil, relu;
  int tiles_x, tiles_per_img, num_patches;   // 8x16 patches: per row, per image, in total (index range [0, num_patches))
  int strip_first, num_strips, strips_per_img, strip_y0;  // 4x32 strips: index range [strip_first, strip_first + num_strips)
  int num_m_tiles, num_n_tiles, cblocks;  // m tile = 2 patches (one per CTA)
  int a_slot_bytes, a_bytes_full, a_bytes_strip, a_slots, b_slots;
  BnAcc* bn_acc;   // STATS kernels only: [2][Cout] accumulators of sum y / sum y^2 over the stored bf16 outputs (train-mode BatchNorm)
};

__device__ __forceinline__ void th_decode_patch(const ConvTc2hArgs& a, int patch, int& b, int& y0, int& x0) {
  if (patch < a.num_patches) {
    b = patch / a.tiles_per_img;
    const int r = patch - b * a.tiles_per_img;
    const int ty = r / a.tiles_x;
    y0 = ty * TH_TILE_H;
    x0 = (r - ty * a.tiles_x) * TH_TILE_W;
  } else if (patch >= a.strip_first && patch < a.strip_first + a.num_strips) {
    const int q = patch - a.strip_first;
    b = q / a.strips_per_img;
    y0 = a.strip_y0;
    x0 = (q - b * a.strips_per_img) * (2 * TH_TILE_W);
  } else {
    b = a.B;  // out of range in the batch dimension: TMA zero fill, stores clipped
    y0 = 0;
    x0 = 0;
  }
}

template <int BLOCK_N, bool STATS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TH_THREADS, 1)
conv_tc2h_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                 const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_res,
                 const __grid_constant__ CUtensorMap map_xs, const __grid_constant__ CUtensorMap map_ys,
                 const __grid_constant__ CUtensorMap map_ress, const ConvTc2hArgs a) {
  constexpr int HALF_N = BLOCK_N / 2;
  constexpr int B_BYTES = HALF_N * 128;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const int NA = a.a_slots, NB = a.b_slots;
  uint8_t* sA = smem;
  uint8_t* sB = sA + NA * a.a_slot_bytes;
  uint8_t* staging = sB + NB * B_BYTES;  // 3 x [128 rows][128 B], 1024-aligned
  uint64_t* a_full = reinterpret_cast<uint64_t*>(staging + TH_STAGING_BYTES);
  uint64_t* a_empty = a_full + TH_MAX_A;
  uint64_t* b_full = a_empty + TH_MAX_A;
  uint64_t* b_empty = b_full + TH_MAX_B;
  uint64_t* tmem_full_bar = b_empty + TH_MAX_B;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint64_t* res_bar = tmem_empty_bar + 2;  // [3]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(res_bar + 3);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int total_tiles = a.num_m_tiles * a.num_n_tiles;

  ptx::griddep_launch_dependents();  // the next kernel's CTAs may take over SMs as ours exit (its prologue overlaps our tail)
  ptx::cluster_sync_all();
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
    ptx::prefetch_tensormap(&map_y);
    if (a.residual) ptx::prefetch_tensormap(&map_res);
    if (a.num_strips > 0) {
      ptx::prefetch_tensormap(&map_xs);
      ptx::prefetch_tensormap(&map_ys);
      if (a.residual) ptx::prefetch_tensormap(&map_ress);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < TH_MAX_A; ++i) {
      ptx::mbar_init(&a_full[i], 2);
      ptx::mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < TH_MAX_B; ++i) {
      ptx::mbar_init(&b_full[i], 2);
      ptx::mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], 2 * TH_EPI_THREADS);  // both CTAs' epilogue threads
    }
    for (int i = 0; i < 3; ++i) ptx::mbar_init(&res_bar[i], 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc2(tmem_ptr_smem, 2 * BLOCK_N);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs; whole warp waits, one elected lane issues) =====================
    ptx::griddep_wait();  // the previous kernel's output (our input) is complete and visible
    uint32_t as = 0, aph = 0, bs = 0, bph = 0;
    for (int tile = cluster_id; tile < total_tiles; tile += num_clusters) {
      const int m_tile = tile / a.num_n_tiles, n_tile = tile - m_tile * a.num_n_tiles;
      int b, y0, x0;
      th_decode_patch(a, 2 * m_tile + (int)rank, b, y0, x0);
      const bool strip = 2 * m_tile >= a.strip_first;   // the same for both CTAs of the pair
      const CUtensorMap* mxp = strip ? &map_xs : &map_x;
      const uint32_t a_tx = 2u * (uint32_t)(strip ? a.a_bytes_strip : a.a_bytes_full);
      const int n_row0 = n_tile * BLOCK_N + (int)rank * HALF_N;
      for (int s = 0; s < 3; ++s) {
        for (int cb = 0; cb < a.cblocks; ++cb) {
          ptx::mbar_wait(&a_empty[as], aph ^ 1, 51);
          if (ptx::elect_one_sync()) {
            ptx::tma2_load_4d(sA + as * a.a_slot_bytes, mxp, &a_full[as], cb * 64, x0 + (s - 1) * a.dil, y0 - a.dil, b);
            if (leader) ptx::mbar_arrive_expect_tx(&a_full[as], a_tx);
            else ptx::mbar_arrive_remote(&a_full[as], 0);
          }
          __syncwarp();
          if (++as == (uint32_t)NA) { as = 0; aph ^= 1; }
          for (int r = 0; r < 3; ++r) {
            ptx::mbar_wait(&b_empty[bs], bph ^ 1, 52);
            if (ptx::elect_one_sync()) {
              ptx::tma2_load_2d(sB + bs * B_BYTES, &map_w, &b_full[bs], (r * 3 + s) * a.Cin + cb * 64, n_row0);
              if (leader) ptx::mbar_arrive_expect_tx(&b_full[bs], 2 * B_BYTES);
              else ptx::mbar_arrive_remote(&b_full[bs], 0);
            }
            __syncwarp();
            if (++bs == (uint32_t)NB) { bs = 0; bph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===================== MMA issuer (leader CTA only; whole warp waits, one elected lane issues) =====================
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(256, BLOCK_N);
      uint32_t as = 0, aph = 0, bs = 0, bph = 0, it = 0;
      for (int tile = cluster_id; tile < total_tiles; tile += num_clusters, ++it) {
        const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
        const bool strip = 2 * (tile / a.num_n_tiles) >= a.strip_first;
        const uint32_t tap_bytes = (uint32_t)a.dil * (strip ? 2 * TH_ROW_BYTES : TH_ROW_BYTES);  // one image row of the staged box
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, 53);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        const int groups = 3 * a.cblocks;
        for (int g = 0; g < groups; ++g) {
          ptx::mbar_wait(&a_full[as], aph, 54);
          const uint32_t a_base = ptx::smem_u32(sA + as * a.a_slot_bytes);
          for (int r = 0; r < 3; ++r) {
            ptx::mbar_wait(&b_full[bs], bph, 55);
            ptx::tc_fence_after();
            if (ptx::elect_one_sync()) {
              const uint64_t adesc = ptx::make_smem_desc_sw128(a_base + r * tap_bytes);
              const uint64_t bdesc = ptx::make_smem_desc_sw128(ptx::smem_u32(sB + bs * B_BYTES));
#pragma unroll
              for (int k = 0; k < 4; ++k) ptx::umma2_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (g | r | k) != 0 ? 1u : 0u);
              ptx::umma2_commit_mc(&b_empty[bs]);
              if (r == 2) {
                ptx::umma2_commit_mc(&a_empty[as]);
                if (g == groups - 1) ptx::umma2_commit_mc(&tmem_full_bar[acc]);
              }
            }
            __syncwarp();
            if (++bs == (uint32_t)NB) { bs = 0; bph ^= 1; }
          }
          if (++as == (uint32_t)NA) { as = 0; aph ^= 1; }
        }
      }
      // all remote arrivals of the last two accumulator uses must land before this CTA's barriers go away
      if (it >= 1) { const uint32_t j = it - 1; ptx::mbar_wait(&tmem_empty_bar[j & 1], (j >> 1) & 1, 56); }
      if (it >= 2) { const uint32_t j = it - 2; ptx::mbar_wait(&tmem_empty_bar[j & 1], (j >> 1) & 1, 57); }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, own 128 TMEM lanes; 8 warps = 256 threads, named barrier 1) =====================
    // warp % 4 = TMEM lane quarter (32 rows), (warp - 4) / 4 = which 32 of a chunk's 64 columns (as in conv_tc2_kernel)
    const int q = warp & 3, half = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const bool elected = (warp == 4 && lane == 0);
    const int sw = row & 7;
    constexpr int CHUNKS = BLOCK_N / 64;
    const bool has_res = a.residual != nullptr;
    const int et = (int)threadIdx.x - 128;   // epilogue thread 0..255
    EpiStats stats;
    if (STATS) epi_stats_init(stats, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(a_full) + 512), a.Cout, et);
    ptx::griddep_wait();  // before the first residual load / output store
    uint32_t it = 0, chunk_ctr = 0;
    for (int tile = cluster_id; tile < total_tiles; tile += num_clusters, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const int m_tile = tile / a.num_n_tiles, n_tile = tile - m_tile * a.num_n_tiles;
      int b, y0, x0;
      th_decode_patch(a, 2 * m_tile + (int)rank, b, y0, x0);
      const bool strip = 2 * m_tile >= a.strip_first;
      const CUtensorMap* myp = strip ? &map_ys : &map_y;
      const CUtensorMap* mrp = strip ? &map_ress : &map_res;
      const int n0 = n_tile * BLOCK_N;
      const float* scale = a.scale + n0;
      const float* bias = a.bias + n0;
      int nvalid = 0;   // STATS: how many of this thread's 16 staged rows (16 pixels of one image row) lie inside the image
      if (STATS) {
        const int rg = et >> 5;
        const int yy = y0 + (strip ? rg >> 1 : rg), xx = x0 + (strip ? (rg & 1) * 16 : 0);
        if (b < a.B && yy < a.Ho) nvalid = min(16, max(0, a.Wo - xx));
      }
      auto issue_residual = [&](int chunk, uint32_t ctr) {
        const uint32_t bsel = ctr % 3;
        ptx::mbar_arrive_expect_tx(&res_bar[bsel], 16384);
        ptx::tma_load_4d(staging + bsel * 16384, mrp, &res_bar[bsel], n0 + chunk * 64, x0, y0, b);
      };
      if (elected) {
        ptx::bulk_wait_group_read1();
        if (has_res) issue_residual(0, chunk_ctr);
      }
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase, 58);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
#pragma unroll 1
      for (int chunk = 0; chunk < CHUNKS; ++chunk, ++chunk_ctr) {
        const uint32_t bsel = chunk_ctr % 3;
        uint8_t* my_row = staging + bsel * 16384 + row * 128;
        if (elected) {
          ptx::bulk_wait_group_read1();
          if (has_res && chunk + 1 < CHUNKS) issue_residual(chunk + 1, chunk_ctr + 1);
        }
        ptx::named_bar_sync(1, TH_EPI_THREADS);
        if (STATS) epi_stats_reduce_prev(stats, et);
        uint32_t r0[32];
        ptx::tmem_ld_32x32(taddr + chunk * 64 + half * 32, r0);
        ptx::tmem_ld_wait();
        if (chunk == CHUNKS - 1) {
          ptx::tc_fence_before();
          ptx::mbar_arrive_remote(&tmem_empty_bar[acc], 0);
        }
        if (has_res) ptx::mbar_wait(&res_bar[bsel], (chunk_ctr / 3) & 1, 59);
#pragma unroll
        for (int gg = 0; gg < 4; ++gg) {
          const int g = half * 4 + gg;  // 16-byte slot of the 128-byte row
          const int c = chunk * 64 + g * 8;
          const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale + c));
          const float4 s1 = __ldg(reinterpret_cast<const float4*>(scale + c + 4));
          const float4 t0 = __ldg(reinterpret_cast<const float4*>(bias + c));
          const float4 t1 = __ldg(reinterpret_cast<const float4*>(bias + c + 4));
          const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
          const float bi[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = fmaf(__uint_as_float(r0[gg * 8 + j]), sc[j], bi[j]);
          uint4* slot = reinterpret_cast<uint4*>(my_row + (((g ^ sw) & 7) << 4));
          if (has_res) {
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
        ptx::fence_proxy_async_smem();
        ptx::named_bar_sync(1, TH_EPI_THREADS);
        if (elected) {
          ptx::tma_store_4d(myp, staging + bsel * 16384, n0 + chunk * 64, x0, y0, b);  // clipped outside the image / batch
          ptx::bulk_commit_group();
        }
        if (STATS) epi_stats_chunk(stats, staging + bsel * 16384, et, nvalid, n0 + chunk * 64);
      }
    }
    if (STATS) epi_stats_flush(stats, et, a.Cout, a.bn_acc, [] { ptx::named_bar_sync(1, TH_EPI_THREADS); });
    if (elected) ptx::bulk_wait_group0();
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc2(tmem_base, 2 * BLOCK_N);
  }
}

// Measured per layer shape (B200): dilation 1 and 2 gain at 60x80 (+13 % / +1 %, the wasted half patch row included) and at 120x160
// (+27 % / +6 %); the dilation-4 layer is MMA-bound either way and its 16-row boxes lose 14 % at 120x160, so it stays on the plain
// kernel.
bool conv_tc2h_applicable(const HkConvDesc& d) {
  return d.kh == 3 && d.kw == 3 && d.stride == 1 && d.pad == d.dil && d.out_c % 128 == 0 && d.in_c % 64 == 0 && (d.dil == 1 || d.dil == 2);
}

template <int BLOCK_N, bool STATS>
static int launch_tc2h(const CUtensorMap& mx, const CUtensorMap& mw, const CUtensorMap& my, const CUtensorMap& mres,
                       const CUtensorMap& mxs, const CUtensorMap& mys, const CUtensorMap& mress, ConvTc2hArgs& a, cudaStream_t s) {
  constexpr int B_BYTES = (BLOCK_N / 2) * 128;
  const int stats_bytes = STATS ? epi_stats_smem_bytes(a.Cout) : 0;
  const int budget = 227 * 1024 - 1024 - TH_STAGING_BYTES - 512 - stats_bytes;
  int na = 3, nb = (budget - na * a.a_slot_bytes) / B_BYTES;
  if (nb > TH_MAX_B) {  // room to spare: one more haloed box in flight
    nb = TH_MAX_B;
    if ((budget - nb * B_BYTES) / a.a_slot_bytes >= 4) na = 4;
  }
  if (nb < 3) return fail(HK_ERR_BAD_ARG, "conv(tcgen05,halo): shared memory budget too small");
  a.a_slots = na;
  a.b_slots = nb;
  const int smem = 1024 + na * a.a_slot_bytes + nb * B_BYTES + TH_STAGING_BYTES + 512 + stats_bytes;
  if (int rc = opt_in_smem<conv_tc2h_kernel<BLOCK_N, STATS>>(smem, "conv(tcgen05,halo)")) return rc;
  const int total = a.num_m_tiles * a.num_n_tiles;
  int clusters = sm_count() / 2;
  if (clusters > total) clusters = total;
  cudaError_t le = launch_pdl(conv_tc2h_kernel<BLOCK_N, STATS>, dim3(2 * clusters), dim3(TH_THREADS), (size_t)smem, s, mx, mw, my, mres, mxs, mys,
                              mress, a);
  if (le != cudaSuccess) return fail(HK_ERR_CUDA, "conv_tc2h_kernel: %s", cudaGetErrorString(le));
  return check_launch("conv_tc2h_kernel");
}

int conv_tc2h_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias, const void* residual,
                     void* y, void* bn_acc, cudaStream_t s) {
  // patch geometry: 8x16 patches over the rows that fill whole patch rows, 4x32 strips over a remainder of 1..4 rows (see the header)
  const int rem_rows = d.out_h % TH_TILE_H;
  const bool use_strips = rem_rows >= 1 && rem_rows <= 4 && d.out_h > TH_TILE_H;
  const int tiles_x = ceil_div(d.out_w, TH_TILE_W);
  const int tiles_y = use_strips ? d.out_h / TH_TILE_H : ceil_div(d.out_h, TH_TILE_H);
  const int strips_per_img = use_strips ? ceil_div(d.out_w, 2 * TH_TILE_W) : 0;
  const long long full_all = (long long)tiles_x * tiles_y * d.batch;
  const long long strip_first_ll = (full_all + 1) / 2 * 2;
  const long long strips_all = (long long)strips_per_img * d.batch;
  const long long patches_all = use_strips ? strip_first_ll + strips_all : full_all;
  const int block_n = pick_block_n_pair(d.out_c, (patches_all + 1) / 2);
  const int ktot = 9 * d.in_c;
  const int box_rows = TH_TILE_H + 2 * d.dil;
  const int strip_box_rows = TH_TILE_H / 2 + 2 * d.dil;
  const char* who = "conv(tcgen05,halo)";
  CUtensorMap mx, mw, my, mres;
  if (int rc = tmap_nhwc_bf16(&mx, x, d.batch, d.in_h, d.in_w, d.in_c, TH_TILE_W, box_rows, 1, who, "activations")) return rc;
  if (int rc = tmap_kmajor_bf16(&mw, w, ktot, d.out_c, block_n / 2, who, "weights")) return rc;
  if (int rc = tmap_nhwc_bf16(&my, y, d.batch, d.out_h, d.out_w, d.out_c, TH_TILE_W, TH_TILE_H, 1, who, "output")) return rc;
  mres = my;
  if (residual) {
    if (int rc = tmap_nhwc_bf16(&mres, residual, d.batch, d.out_h, d.out_w, d.out_c, TH_TILE_W, TH_TILE_H, 1, who, "residual")) return rc;
  }
  CUtensorMap mxs = mx, mys = my, mress = mres;   // 4x32 strip flavours of the activation / output / residual maps
  if (use_strips) {
    const int strip_w = 2 * TH_TILE_W, strip_h = TH_TILE_H / 2;
    if (int rc = tmap_nhwc_bf16(&mxs, x, d.batch, d.in_h, d.in_w, d.in_c, strip_w, strip_box_rows, 1, who, "strip activations")) return rc;
    if (int rc = tmap_nhwc_bf16(&mys, y, d.batch, d.out_h, d.out_w, d.out_c, strip_w, strip_h, 1, who, "strip output")) return rc;
    mress = mys;
    if (residual) {
      if (int rc = tmap_nhwc_bf16(&mress, residual, d.batch, d.out_h, d.out_w, d.out_c, strip_w, strip_h, 1, who, "strip residual")) return rc;
    }
  }
  ConvTc2hArgs a;
  a.scale = scale; a.bias = bias;
  a.residual = static_cast<const __nv_bfloat16*>(residual);
  a.B = d.batch; a.Ho = d.out_h; a.Wo = d.out_w; a.Cout = d.out_c; a.Cin = d.in_c; a.pad = d.pad; a.dil = d.dil; a.relu = d.relu;
  a.tiles_x = tiles_x;
  a.tiles_per_img = tiles_x * tiles_y;
  HK_REQUIRE(patches_all < 0x3fffffffLL, "conv(tcgen05,halo): too many tiles");
  a.num_patches = (int)full_all;
  a.strip_first = use_strips ? (int)strip_first_ll : 0x7fffffff;   // no strips: no pair ever reaches the strip range
  a.num_strips = (int)strips_all;
  a.strips_per_img = strips_per_img > 0 ? strips_per_img : 1;
  a.strip_y0 = tiles_y * TH_TILE_H;
  a.num_m_tiles = (int)((patches_all + 1) / 2);
  a.num_n_tiles = d.out_c / block_n;
  a.cblocks = d.in_c / 64;
  a.a_bytes_full = box_rows * TH_ROW_BYTES;
  a.a_bytes_strip = strip_box_rows * 2 * TH_ROW_BYTES;
  a.a_slot_bytes = use_strips && a.a_bytes_strip > a.a_bytes_full ? a.a_bytes_strip : a.a_bytes_full;
  a.bn_acc = static_cast<BnAcc*>(bn_acc);
  if (bn_acc) return block_n == 256 ? launch_tc2h<256, true>(mx, mw, my, mres, mxs, mys, mress, a, s) : launch_tc2h<128, true>(mx, mw, my, mres, mxs, mys, mress, a, s);
  return block_n == 256 ? launch_tc2h<256, false>(mx, mw, my, mres, mxs, mys, mress, a, s) : launch_tc2h<128, false>(mx, mw, my, mres, mxs, mys, mress, a, s);
}

}  // namespace hk
