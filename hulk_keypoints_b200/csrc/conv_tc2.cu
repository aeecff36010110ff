// 2-CTA (cta_group::2) tcgen05 implicit-GEMM convolution: the CTA PAIR of one TPC computes a 256-pixel x BLOCK_N tile.
//
// Same math and data path as conv_tc_kernel (TMA tap-shifted boxes of the NHWC activation as A, K-major weights
// as B, TMEM accumulators, fused scale/bias/residual/ReLU epilogue), but one tcgen05.mma.cta_group::2 (M=256) is
// issued by the leader CTA for both SMs: each CTA stages its own 128 rows of A and only HALF of the weight tile
// (BLOCK_N/2 rows); the tensor cores exchange the B halves over the pair's private path.  Per CTA that cuts the
// shared-memory operand reads from (4 KB + 32*N B) to (4 KB + 16*N B) per K=16 step and halves the L2->SM weight
// traffic -- the two things that bound the 1-CTA kernel (SS-mode MMA at N=256 needs ~96 B/clk of smem reads; measured
// sustain is ~85 B/clk, i.e. 88 % tensor-pipe activity; N=128 needs 128 B/clk).
//
// Protocol (per stage s, accumulator buffer a):
//   full[s]       lives in the LEADER's smem, 2 arrivals (both producers) + 2x STAGE_BYTES of TMA transaction bytes;
//                 both CTAs issue cp.async.bulk.tensor...cta_group::2 whose completion is routed to the leader's barrier
//   empty[s]      one per CTA; tcgen05.commit.cta_group::2...multicast::cluster arrives on both when the MMAs retire
//   tmem_full[a]  one per CTA (multicast commit); each CTA's epilogue drains its own 128 TMEM lanes
//   tmem_empty[a] in the leader, 2 x 128 arrivals (the peer's epilogue threads arrive remotely via mapa)
//
// Epilogue through shared memory and TMA (64-channel chunks, three 16 KB staging buffers per CTA): the residual chunk is
// TMA-loaded into the swizzled staging buffer one chunk ahead, each thread fixes up its own row in place (conflict-free
// with the 128-byte swizzle) and one elected thread issues the TMA stores.  The direct version (16-byte accesses at a
// >= 256-byte lane stride) cost 32 L1 wavefronts per warp instruction and made the 1x1 downsample convs and the
// N=128 layer epilogue-bound.
//
// DS = true ("block entry", reference src/resnet.py:56-58 + :64-65,184-188): the 1x1 downsample conv of a stride/channel-changing
// BasicBlock reads exactly the centre tap of conv1's activation operand (pad = dil*(k/2): tap offset 0, same stride), so both convs
// run in ONE launch.  Every (m, n) work item is two accumulator uses: sub 0 = conv1 (kh*kw*cblocks K blocks, scale/bias/ReLU, y),
// sub 1 = downsample (cblocks K blocks of the centre-tap boxes against the 1x1 weights, scale2/bias2, no ReLU, y2).  The barrier
// protocol is unchanged (sub-tiles simply take consecutive accumulator turns); sub 1's epilogue hides under the next item's conv1
// mainloop.  Sub 0's epilogue would otherwise hold its accumulator through the short sub-1 mainloop and stall the next conv1, so in
// DS mode it drains all of its TMEM columns into packed bf16 registers first, releases the accumulator, and only then stages/stores.
//
// HEAD = true (the network's LAST conv, reference src/resnet.py:60-67 of layer4[2] + the 1x1 scoring conv `fc` at :215 restricted to the K
// live rows of src/model.py:21): the feature map is consumed by nothing but that 1x1 conv, so the epilogue multiplies its finished rows
// (conv + BN + shortcut + ReLU, rounded to bf16 exactly as they would have been stored) with the K x Cout scoring weights and adds the
// K partial logits of each pixel to the (B,K,Ho,Wo) fp32 logits -- the (B,Ho,Wo,512) feature map is never written, and the stand-alone
// head_logits_kernel (one full read of it) disappears.  Each pixel receives exactly two contributions (the two 256-column N tiles) on a
// zero-initialised buffer, and fp32 addition is commutative, so the result does not depend on their order.
#include <cuda.h>
#include <stdlib.h>

#include "hk_common.cuh"
#include "hk_bn_acc.cuh"
#include "hk_ptx.cuh"
#include "hk_ptx2.cuh"

namespace hk {

constexpr int T2_BOX_H = 4, T2_BOX_W = 16;
constexpr int T2_BOX_BYTES = 64 * 128;   // 8 KB: 64 pixels x 64 ch bf16
constexpr int T2_A_BYTES = 2 * T2_BOX_BYTES;  // 128 rows per CTA
constexpr int T2_THREADS = 384;      // warps 0-3: TMA producer, MMA issuer, TMEM allocator, spare; warps 4-11: epilogue
constexpr int T2_EPI_THREADS = 256;

struct ConvTc2Args {
  const float* scale;
  const float* bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* y;
  int B, Ho, Wo, Cout;
  int Cin, kh, kw, stride, pad, dil, relu;
  int tiles_x, tiles_per_img, num_boxes;
  int num_m_tiles, num_n_tiles, cblocks;  // m tiles of 256 pixels (4 boxes)
  const float* scale2;   // DS kernels only: folded BN of the 1x1 downsample conv, ReLU flag of its epilogue (0 in the reference)
  const float* bias2;
  int relu2, early_release, s_major;
  const float* head_w;   // HEAD kernels only: (head_k, Cout) fp32 scoring weights, (head_k) bias, (B, head_k, Ho, Wo) fp32 logits (zero on entry)
  const float* head_b;
  float* head_logits;
  int head_k;
  BnAcc* bn_acc;         // STATS kernels only: [2][Cout] accumulators of sum y / sum y^2 over the stored bf16 outputs (train-mode BatchNorm)
#ifdef HK_DIAG  // diagnostics build only (python -m hulk_keypoints_b200.build --diag -> libhulk_sm100_diag.so); never in the shipped library
  int dbg_mode;    // HK_TC2_DEBUG bit flags: 1 = skip the MMAs, 2 = skip the TMA operand loads, 4 = skip the epilogue body (results are garbage)
  long long* dbg;  // optional timeline of cluster 0's leader CTA (tools/diag_tc2_timeline.py)
#endif
};
#ifdef HK_DIAG
#define T2_DBG_MODE(a) ((a).dbg_mode)
#define T2_STAMP(role, t, slot) \
  do { if (a.dbg && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (t) < 16) a.dbg[((role) * 16 + (t)) * 8 + (slot)] = clock64(); } while (0)
#else
#define T2_DBG_MODE(a) 0
#define T2_STAMP(role, t, slot) do { } while (0)
#endif

template <int BLOCK_N>
struct Tc2Cfg {
  static constexpr int HALF_N = BLOCK_N / 2;
  static constexpr int B_BYTES = HALF_N * 128;
  static constexpr int STAGE_BYTES = T2_A_BYTES + B_BYTES;
  static constexpr int STAGING_BUFS = 3;               // chunk c uses buffer c % 3: its previous user is 3 chunks old
  static constexpr int STAGING_BYTES = STAGING_BUFS * 128 * 128;  // 128-row x 64-channel bf16 chunk buffers
  static constexpr int STAGES = (160 * 1024) / STAGE_BYTES > 8 ? 8 : (160 * 1024) / STAGE_BYTES;  // 5 (N=256) / 6 (N=128)
  static constexpr int TMEM_COLS = 2 * BLOCK_N;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + 1024 + 256;
};


__device__ __forceinline__ void t2_decode_box(const ConvTc2Args& a, int box, int& b, int& y0, int& x0) {
  if (box < a.num_boxes) {
    b = box / a.tiles_per_img;
    const int r = box - b * a.tiles_per_img;
    const int ty = r / a.tiles_x;
    y0 = ty * T2_BOX_H;
    x0 = (r - ty * a.tiles_x) * T2_BOX_W;
  } else {
    b = a.B;  // out of range in the batch dimension: TMA zero fill, stores masked
    y0 = 0;
    x0 = 0;
  }
}

constexpr int T2_HEAD_MAX_K = 8;
constexpr int T2_HEAD_SMEM_BYTES = T2_HEAD_MAX_K * 256 * 4 + 128 * T2_HEAD_MAX_K * 4;   // weight slice of one N tile + the half-row exchange

template <int BLOCK_N, bool DS, bool STATS, bool HEAD = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(T2_THREADS, 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_res,
                const __grid_constant__ CUtensorMap map_w2, const __grid_constant__ CUtensorMap map_y2, const ConvTc2Args a) {
  constexpr int NSUB = DS ? 2 : 1;
  using Cfg = Tc2Cfg<BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* staging = smem + STAGES * Cfg::STAGE_BYTES;  // 3 x [128 rows][128 B], 1024-aligned
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + Cfg::STAGING_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint64_t* res_bar = tmem_empty_bar + 2;  // [3]: residual chunk landed in staging buffer i
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(res_bar + 3);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp: provably uniform
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int total_tiles = a.num_m_tiles * a.num_n_tiles;
  const int num_kb = a.kh * a.kw * a.cblocks;

  ptx::griddep_launch_dependents();  // the next kernel's CTAs may take over SMs as ours exit (its prologue overlaps our tail)
  ptx::cluster_sync_all();
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
    ptx::prefetch_tensormap(&map_y);
    if (a.residual) ptx::prefetch_tensormap(&map_res);
    if (DS) {
      ptx::prefetch_tensormap(&map_w2);
      ptx::prefetch_tensormap(&map_y2);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      ptx::mbar_init(&full_bar[i], 2);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], 2 * T2_EPI_THREADS);  // both CTAs' epilogue threads
    }
    for (int i = 0; i < 3; ++i) ptx::mbar_init(&res_bar[i], 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc2(tmem_ptr_smem, Cfg::TMEM_COLS);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    {
      // ===================== TMA producer (both CTAs; whole warp waits, one elected lane issues) =====================
      ptx::griddep_wait();  // the previous kernel's output (our input) is complete and visible
      uint32_t stage = 0, phase = 0, pit = 0;
      for (int tile = cluster_id; tile < total_tiles; tile += num_clusters, ++pit) {
        const int m_tile = tile / a.num_n_tiles, n_tile = tile - m_tile * a.num_n_tiles;
        int b0, y0, x0, b1, y1, x1;
        T2_STAMP(0, pit, 0);
        t2_decode_box(a, 4 * m_tile + 2 * (int)rank, b0, y0, x0);
        t2_decode_box(a, 4 * m_tile + 2 * (int)rank + 1, b1, y1, x1);
        const int n_row0 = n_tile * BLOCK_N + (int)rank * Cfg::HALF_N;
        if (DS && a.s_major) {
          // K blocks in the haloed kernel's order (s, channel block, r): the fp32 accumulation sequence -- and therefore every output
          // bit -- matches conv_tc2h_kernel, which is where this conv runs when it is launched on its own
          for (int s = 0; s < a.kw; ++s) {
            for (int cb = 0; cb < a.cblocks; ++cb) {
              for (int r = 0; r < a.kh; ++r) {
                const int dy = r * a.dil - a.pad, dx = s * a.dil - a.pad;
                const int kbase = (r * a.kw + s) * a.Cin;
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 31);
                if (ptx::elect_one_sync()) {
                  uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                  ptx::tma2_load_4d(sa, &map_x, &full_bar[stage], cb * 64, x0 * a.stride + dx, y0 * a.stride + dy, b0);
                  ptx::tma2_load_4d(sa + T2_BOX_BYTES, &map_x, &full_bar[stage], cb * 64, x1 * a.stride + dx, y1 * a.stride + dy, b1);
                  ptx::tma2_load_2d(sa + T2_A_BYTES, &map_w, &full_bar[stage], kbase + cb * 64, n_row0);
                  if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
                  else ptx::mbar_arrive_remote(&full_bar[stage], 0);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
              }
            }
          }
        } else
        for (int r = 0; r < a.kh; ++r) {
          for (int s = 0; s < a.kw; ++s) {
            const int dy = r * a.dil - a.pad, dx = s * a.dil - a.pad;
            const int kbase = (r * a.kw + s) * a.Cin;
            for (int cb = 0; cb < a.cblocks; ++cb) {
              if (T2_DBG_MODE(a) & 2) continue;
              ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 31);
              if (ptx::elect_one_sync()) {
                uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                ptx::tma2_load_4d(sa, &map_x, &full_bar[stage], cb * 64, x0 * a.stride + dx, y0 * a.stride + dy, b0);
                ptx::tma2_load_4d(sa + T2_BOX_BYTES, &map_x, &full_bar[stage], cb * 64, x1 * a.stride + dx, y1 * a.stride + dy, b1);
                ptx::tma2_load_2d(sa + T2_A_BYTES, &map_w, &full_bar[stage], kbase + cb * 64, n_row0);
                if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
                else ptx::mbar_arrive_remote(&full_bar[stage], 0);
              }
              __syncwarp();
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
          }
        }
        if (DS) {  // sub 1: the 1x1 downsample conv = centre tap (offset 0) of the same boxes against its own weights
          const int cdy = (a.kh >> 1) * a.dil - a.pad, cdx = (a.kw >> 1) * a.dil - a.pad;
          for (int cb = 0; cb < a.cblocks; ++cb) {
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 31);
            if (ptx::elect_one_sync()) {
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              ptx::tma2_load_4d(sa, &map_x, &full_bar[stage], cb * 64, x0 * a.stride + cdx, y0 * a.stride + cdy, b0);
              ptx::tma2_load_4d(sa + T2_BOX_BYTES, &map_x, &full_bar[stage], cb * 64, x1 * a.stride + cdx, y1 * a.stride + cdy, b1);
              ptx::tma2_load_2d(sa + T2_A_BYTES, &map_w2, &full_bar[stage], cb * 64, n_row0);
              if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
              else ptx::mbar_arrive_remote(&full_bar[stage], 0);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        T2_STAMP(0, pit, 1);
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===================== MMA issuer (leader CTA only; whole warp waits, one elected lane issues) =====================
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(256, BLOCK_N);
      uint32_t stage = 0, phase = 0, it = 0;
      for (int tile = cluster_id; tile < total_tiles; tile += num_clusters) {
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub, ++it) {
          const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
          const int nkb = sub ? a.cblocks : num_kb;
          T2_STAMP(1, it, 0);
          ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, 32);
          ptx::tc_fence_after();
          T2_STAMP(1, it, 1);
          const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
          for (int kb = 0; kb < nkb; ++kb) {
            if (!(T2_DBG_MODE(a) & 2)) ptx::mbar_wait(&full_bar[stage], phase, 33);
            if (kb == 0) T2_STAMP(1, it, 2);
            ptx::tc_fence_after();
            const uint32_t sa = ptx::smem_u32(smem + stage * Cfg::STAGE_BYTES);
            const uint64_t adesc = ptx::make_smem_desc_sw128(sa);
            const uint64_t bdesc = ptx::make_smem_desc_sw128(sa + T2_A_BYTES);
            if (ptx::elect_one_sync()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (!(T2_DBG_MODE(a) & 1)) ptx::umma2_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              ptx::umma2_commit_mc(&empty_bar[stage]);
              if (kb == nkb - 1) ptx::umma2_commit_mc(&tmem_full_bar[acc]);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          T2_STAMP(1, it, 3);
        }
      }
      // all remote arrivals of the last two accumulator uses must land before this CTA's barriers go away
      if (it >= 1) { const uint32_t j = it - 1; ptx::mbar_wait(&tmem_empty_bar[j & 1], (j >> 1) & 1, 34); }
      if (it >= 2) { const uint32_t j = it - 2; ptx::mbar_wait(&tmem_empty_bar[j & 1], (j >> 1) & 1, 35); }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, own 128 TMEM lanes; 8 warps = 256 threads, named barrier 1) =====================
    // warp % 4 = TMEM lane quarter (32 rows), (warp - 4) / 4 = which 32 of a chunk's 64 columns: with 4 warps the drain of a 256-column
    // tile took ~6k clocks, which capped the output-heavy 1x1 downsample convs (K = 64..256) at ~3 TB/s of stores
    const int q = warp & 3, half = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const bool elected = (warp == 4 && lane == 0);
    const int sw = row & 7;
    constexpr int CHUNKS = BLOCK_N / 64;
    const int et = (int)threadIdx.x - 128;   // epilogue thread 0..255
    EpiStats stats;
    if (STATS) epi_stats_init(stats, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256), a.Cout, et);
    int head_loaded = -1;   // HEAD: N tile whose scoring-weight slice is in shared memory
    ptx::griddep_wait();  // before the first residual load / output store
    uint32_t it = 0, chunk_ctr = 0;      // chunk_ctr selects the staging buffer and the res_bar phase
    for (int tile = cluster_id; tile < total_tiles; tile += num_clusters) {
      const int m_tile = tile / a.num_n_tiles, n_tile = tile - m_tile * a.num_n_tiles;
      int b0, y0, x0, b1, y1, x1;          // this CTA's two 4x16 boxes (64 rows each)
      t2_decode_box(a, 4 * m_tile + 2 * (int)rank, b0, y0, x0);
      t2_decode_box(a, 4 * m_tile + 2 * (int)rank + 1, b1, y1, x1);
      const int n0 = n_tile * BLOCK_N;
      int nvalid = 0;   // STATS: how many of this thread's 16 staged rows (one image row of one box) lie inside the image
      if (STATS) {
        const int rg = et >> 5, second = rg >> 2;
        const int bb = second ? b1 : b0, yy = (second ? y1 : y0) + (rg & 3), xx = second ? x1 : x0;
        if (bb < a.B && yy < a.Ho) nvalid = min(16, max(0, a.Wo - xx));
      }
#pragma unroll
      for (int sub = 0; sub < NSUB; ++sub, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const float* scale = (sub ? a.scale2 : a.scale) + n0;
      const float* bias = (sub ? a.bias2 : a.bias) + n0;
      const int relu = sub ? a.relu2 : a.relu;
      const CUtensorMap* myp = sub ? &map_y2 : &map_y;
      const bool has_res = !DS && a.residual != nullptr;   // the block-entry kernels carry no shortcut operand

      // elected thread only.  wait_group.read 1 = every TMA store but the newest has finished reading smem, so the buffers
      // of chunks ctr-2 and older -- i.e. (ctr+1) % 3 and ctr % 3 -- are free.
      auto issue_residual = [&](int chunk, uint32_t ctr) {
        const uint32_t bsel = ctr % 3;
        uint8_t* buf = staging + bsel * 16384;
        ptx::mbar_arrive_expect_tx(&res_bar[bsel], 16384);
        ptx::tma_load_4d(buf, &map_res, &res_bar[bsel], n0 + chunk * 64, x0, y0, b0);
        ptx::tma_load_4d(buf + 8192, &map_res, &res_bar[bsel], n0 + chunk * 64, x1, y1, b1);
      };
      if (elected) {
        T2_STAMP(2, it, 0);
        ptx::bulk_wait_group_read1();
        if (has_res) issue_residual(0, chunk_ctr);
      }
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase, 36);
      ptx::tc_fence_after();
      if (elected) T2_STAMP(2, it, 1);
      if (T2_DBG_MODE(a) & 4) {
        ptx::tc_fence_before();
        ptx::mbar_arrive_remote(&tmem_empty_bar[acc], 0);
        continue;
      }
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
      if (DS && sub == 0 && a.early_release) {
        // drain the whole accumulator first (affine + ReLU + bf16 pack in registers), hand it back to the MMA warp, then stage and store
        uint32_t pk[CHUNKS][16];
#pragma unroll
        for (int chunk = 0; chunk < CHUNKS; ++chunk) {
          uint32_t r0[32];
          ptx::tmem_ld_32x32(taddr + chunk * 64 + half * 32, r0);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int gg = 0; gg < 4; ++gg) {
            const int c = chunk * 64 + (half * 4 + gg) * 8;
            const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale + c));
            const float4 s1 = __ldg(reinterpret_cast<const float4*>(scale + c + 4));
            const float4 t0 = __ldg(reinterpret_cast<const float4*>(bias + c));
            const float4 t1 = __ldg(reinterpret_cast<const float4*>(bias + c + 4));
            const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
            const float bi[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              v[j] = fmaf(__uint_as_float(r0[gg * 8 + j]), sc[j], bi[j]);
              if (relu) v[j] = fmaxf(v[j], 0.f);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) pk[chunk][gg * 4 + j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
          }
        }
        ptx::tc_fence_before();
        ptx::mbar_arrive_remote(&tmem_empty_bar[acc], 0);
#pragma unroll
        for (int chunk = 0; chunk < CHUNKS; ++chunk, ++chunk_ctr) {
          const uint32_t bsel = chunk_ctr % 3;
          uint8_t* my_row = staging + bsel * 16384 + row * 128;
          if (elected) ptx::bulk_wait_group_read1();
          ptx::named_bar_sync(1, T2_EPI_THREADS);  // staging[bsel] is free for everybody
#pragma unroll
          for (int gg = 0; gg < 4; ++gg) {
            const int g = half * 4 + gg;
            *reinterpret_cast<uint4*>(my_row + (((g ^ sw) & 7) << 4)) =
                make_uint4(pk[chunk][gg * 4], pk[chunk][gg * 4 + 1], pk[chunk][gg * 4 + 2], pk[chunk][gg * 4 + 3]);
          }
          ptx::fence_proxy_async_smem();
          ptx::named_bar_sync(1, T2_EPI_THREADS);
          if (elected) {
            const uint8_t* buf = staging + bsel * 16384;
            ptx::tma_store_4d(myp, buf, n0 + chunk * 64, x0, y0, b0);
            ptx::tma_store_4d(myp, buf + 8192, n0 + chunk * 64, x1, y1, b1);
            ptx::bulk_commit_group();
          }
        }
        continue;
      }
      if (HEAD) {
        // ---- last conv of the network: rows go straight into the K scoring dot products, nothing is stored ----
        float* hw = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);   // [head_k][256]: scoring weights of this N tile
        float* hx = hw + T2_HEAD_MAX_K * 256;                                                  // [128 rows][head_k]: upper-half partial sums
        const int K = a.head_k;
        if (n_tile != head_loaded) {   // cluster-uniform (in practice once: the cluster stride is even, so a cluster keeps its N tile)
          ptx::named_bar_sync(1, T2_EPI_THREADS);   // nobody still reads the previous slice
          for (int i = et; i < K * 256; i += T2_EPI_THREADS) hw[i] = __ldg(a.head_w + (size_t)(i >> 8) * a.Cout + n0 + (i & 255));
          head_loaded = n_tile;                      // visible to everybody after the first chunk's barrier
        }
        float p[T2_HEAD_MAX_K];
#pragma unroll
        for (int k = 0; k < T2_HEAD_MAX_K; ++k) p[k] = 0.f;
#pragma unroll 1
        for (int chunk = 0; chunk < CHUNKS; ++chunk, ++chunk_ctr) {
          const uint32_t bsel = chunk_ctr % 3;
          const uint8_t* my_row = staging + bsel * 16384 + row * 128;
          // one barrier per chunk: everybody has finished chunk-1, hence the reads of the buffer the elected thread refills next
          ptx::named_bar_sync(1, T2_EPI_THREADS);
          if (elected && has_res && chunk + 1 < CHUNKS) issue_residual(chunk + 1, chunk_ctr + 1);
          uint32_t r0[32];
          ptx::tmem_ld_32x32(taddr + chunk * 64 + half * 32, r0);
          ptx::tmem_ld_wait();
          if (chunk == CHUNKS - 1) {
            ptx::tc_fence_before();
            ptx::mbar_arrive_remote(&tmem_empty_bar[acc], 0);
          }
          if (has_res) ptx::mbar_wait(&res_bar[bsel], (chunk_ctr / 3) & 1, 37);
#pragma unroll
          for (int gg = 0; gg < 4; ++gg) {
            const int g = half * 4 + gg;
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
            if (has_res) {
              const uint4 rr = *reinterpret_cast<const uint4*>(my_row + (((g ^ sw) & 7) << 4));
              float lo, hi;
              unpack_bf16x2(rr.x, lo, hi); v[0] += lo; v[1] += hi;
              unpack_bf16x2(rr.y, lo, hi); v[2] += lo; v[3] += hi;
              unpack_bf16x2(rr.z, lo, hi); v[4] += lo; v[5] += hi;
              unpack_bf16x2(rr.w, lo, hi); v[6] += lo; v[7] += hi;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (relu) v[j] = fmaxf(v[j], 0.f);
              v[j] = __bfloat162float(__float2bfloat16_rn(v[j]));   // the value the feature map would have held
            }
#pragma unroll
            for (int k = 0; k < T2_HEAD_MAX_K; ++k) {
              if (k < K) {
                const float4 w0 = *reinterpret_cast<const float4*>(hw + k * 256 + c);       // same address for the whole warp: broadcast
                const float4 w1 = *reinterpret_cast<const float4*>(hw + k * 256 + c + 4);
                float acc_k = p[k];
                acc_k = fmaf(v[0], w0.x, acc_k); acc_k = fmaf(v[1], w0.y, acc_k); acc_k = fmaf(v[2], w0.z, acc_k); acc_k = fmaf(v[3], w0.w, acc_k);
                acc_k = fmaf(v[4], w1.x, acc_k); acc_k = fmaf(v[5], w1.y, acc_k); acc_k = fmaf(v[6], w1.z, acc_k); acc_k = fmaf(v[7], w1.w, acc_k);
                p[k] = acc_k;
              }
            }
          }
        }
        // the two 32-column halves of a row live in different warps: the upper half hands its sums over, the lower half finishes the pixel
        if (half == 1) {
#pragma unroll
          for (int k = 0; k < T2_HEAD_MAX_K; ++k)
            if (k < K) hx[row * T2_HEAD_MAX_K + k] = p[k];
        }
        ptx::named_bar_sync(1, T2_EPI_THREADS);
        if (half == 0) {
          const int second = row >> 6, rr = row & 63;
          const int pb = second ? b1 : b0, py = (second ? y1 : y0) + (rr >> 4), px = (second ? x1 : x0) + (rr & 15);
          if (pb < a.B && py < a.Ho && px < a.Wo) {
            float* dst = a.head_logits + (((size_t)pb * K) * a.Ho + py) * a.Wo + px;
#pragma unroll
            for (int k = 0; k < T2_HEAD_MAX_K; ++k)
              if (k < K) atomicAdd(dst + (size_t)k * a.Ho * a.Wo, p[k] + hx[row * T2_HEAD_MAX_K + k] + (n_tile == 0 ? __ldg(a.head_b + k) : 0.f));
          }
        }
        continue;
      }
#pragma unroll 1
      for (int chunk = 0; chunk < CHUNKS; ++chunk, ++chunk_ctr) {
        const uint32_t bsel = chunk_ctr % 3;
        uint8_t* my_row = staging + bsel * 16384 + row * 128;
        if (elected) {
          ptx::bulk_wait_group_read1();
          if (has_res && chunk + 1 < CHUNKS) issue_residual(chunk + 1, chunk_ctr + 1);  // one chunk ahead
        }
        ptx::named_bar_sync(1, T2_EPI_THREADS);  // staging[bsel] is free for everybody (elected passed its wait_group)
        if (STATS) epi_stats_reduce_prev(stats, et);
        if (elected && chunk == 0) T2_STAMP(2, it, 2);
        uint32_t r0[32];
        ptx::tmem_ld_32x32(taddr + chunk * 64 + half * 32, r0);
        ptx::tmem_ld_wait();
        if (elected && chunk == 0) T2_STAMP(2, it, 3);
        if (chunk == CHUNKS - 1) {  // accumulator fully drained: release it to the MMA warp
          ptx::tc_fence_before();
          ptx::mbar_arrive_remote(&tmem_empty_bar[acc], 0);
        }
        if (has_res) ptx::mbar_wait(&res_bar[bsel], (chunk_ctr / 3) & 1, 37);
        if (elected && chunk == 0) T2_STAMP(2, it, 4);
#pragma unroll
        for (int gg = 0; gg < 4; ++gg) {
          const int g = half * 4 + gg;     // 16-byte slot of the 128-byte row
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
          uint4* slot = reinterpret_cast<uint4*>(my_row + (((g ^ sw) & 7) << 4));  // 128-byte swizzle, as TMA expects
          if (has_res) {
            const uint4 rr = *slot;
            float lo, hi;
            unpack_bf16x2(rr.x, lo, hi); v[0] += lo; v[1] += hi;
            unpack_bf16x2(rr.y, lo, hi); v[2] += lo; v[3] += hi;
            unpack_bf16x2(rr.z, lo, hi); v[4] += lo; v[5] += hi;
            unpack_bf16x2(rr.w, lo, hi); v[6] += lo; v[7] += hi;
          }
          if (relu) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          *slot = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        }
        ptx::fence_proxy_async_smem();
        if (elected && chunk == 0) T2_STAMP(2, it, 5);
        ptx::named_bar_sync(1, T2_EPI_THREADS);
        if (elected && chunk == 0) T2_STAMP(2, it, 6);
        if (elected && chunk == CHUNKS - 1) T2_STAMP(2, it, 7);
        if (elected) {
          const uint8_t* buf = staging + bsel * 16384;
          ptx::tma_store_4d(myp, buf, n0 + chunk * 64, x0, y0, b0);         // clipped outside the image / batch
          ptx::tma_store_4d(myp, buf + 8192, n0 + chunk * 64, x1, y1, b1);
          ptx::bulk_commit_group();
        }
        if (STATS) epi_stats_chunk(stats, staging + bsel * 16384, et, nvalid, n0 + chunk * 64);
      }
      }
    }
    if (STATS) epi_stats_flush(stats, et, a.Cout, a.bn_acc, [] { ptx::named_bar_sync(1, T2_EPI_THREADS); });
    if (elected) ptx::bulk_wait_group0();
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
  }
}

#ifdef HK_DIAG
static long long* g_tc2_dbg = nullptr;
extern "C" __attribute__((visibility("default"))) void hk_debug_set_tc2_timeline(long long* dev_buf) { g_tc2_dbg = dev_buf; }
#endif

bool conv_tc2h_applicable(const HkConvDesc& d);

bool conv_tc2_applicable(const HkConvDesc& d) {
  static const bool disabled = getenv("HK_DISABLE_2CTA") != nullptr;
  return !disabled && d.out_c % 128 == 0 && d.in_c % 64 == 0 && (d.stride == 1 || d.stride == 2);
}

template <int BLOCK_N, bool DS, bool STATS, bool HEAD = false>
static int launch_tc2(const CUtensorMap& mx, const CUtensorMap& mw, const CUtensorMap& my, const CUtensorMap& mres,
                      const CUtensorMap& mw2, const CUtensorMap& my2, const ConvTc2Args& a, cudaStream_t s) {
  using Cfg = Tc2Cfg<BLOCK_N>;
  const int smem_bytes = Cfg::SMEM_BYTES + (STATS ? epi_stats_smem_bytes(a.Cout) : 0) + (HEAD ? T2_HEAD_SMEM_BYTES : 0);
  if (smem_bytes > 227 * 1024) return fail(HK_ERR_BAD_ARG, "conv(tcgen05,2cta): %d bytes of shared memory needed", smem_bytes);
  if (int rc = opt_in_smem<conv_tc2_kernel<BLOCK_N, DS, STATS, HEAD>>(smem_bytes, "conv(tcgen05,2cta)")) return rc;
  const int total = a.num_m_tiles * a.num_n_tiles;
  int clusters = sm_count() / 2;
  if (clusters > total) clusters = total;
  cudaError_t le = launch_pdl(conv_tc2_kernel<BLOCK_N, DS, STATS, HEAD>, dim3(2 * clusters), dim3(T2_THREADS), (size_t)smem_bytes, s, mx, mw, my, mres,
                              mw2, my2, a);
  if (le != cudaSuccess) return fail(HK_ERR_CUDA, "conv_tc2_kernel: %s", cudaGetErrorString(le));
  return check_launch("conv_tc2_kernel");
}

// ds != nullptr: block-entry launch (conv1 + the 1x1 downsample conv of the same input, see the header)
struct ConvTc2Head {
  const float* w;      // (K, Cout) fp32
  const float* b;      // (K)
  float* logits;       // (B, K, Ho, Wo) fp32, zero on entry
  int K;
};

struct ConvTc2Ds {
  const void* w;       // (Cout, Cin) bf16, K-major
  const float* scale;
  const float* bias;
  void* y;             // (B, Ho, Wo, Cout) bf16
  int relu;
};

static int conv_tc2_launch_impl(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                                const void* residual, void* y, const ConvTc2Ds* ds, void* bn_acc, cudaStream_t s,
                                const ConvTc2Head* head = nullptr) {
  const long long boxes_all = (long long)ceil_div(d.out_w, T2_BOX_W) * ceil_div(d.out_h, T2_BOX_H) * d.batch;
  // HEAD: 256-column tiles always -- exactly two N tiles (Cout = 512) must add into every logit for the sum to be order-independent
  const int block_n = head ? 256 : pick_block_n_pair(d.out_c, (boxes_all + 3) / 4);
  const int ktot = d.kh * d.kw * d.in_c;
  const char* who = "conv(tcgen05,2cta)";
  CUtensorMap mx, mw, my, mres;
  if (int rc = tmap_nhwc_bf16(&mx, x, d.batch, d.in_h, d.in_w, d.in_c, T2_BOX_W, T2_BOX_H, d.stride, who, "activations")) return rc;
  if (int rc = tmap_kmajor_bf16(&mw, w, ktot, d.out_c, block_n / 2, who, "weights")) return rc;
  // HEAD: nothing is stored; the output map only has to be well-formed
  if (int rc = tmap_nhwc_bf16(&my, y ? y : residual, d.batch, d.out_h, d.out_w, d.out_c, T2_BOX_W, T2_BOX_H, 1, who, "output")) return rc;
  mres = my;
  if (residual) {
    if (int rc = tmap_nhwc_bf16(&mres, residual, d.batch, d.out_h, d.out_w, d.out_c, T2_BOX_W, T2_BOX_H, 1, who, "residual")) return rc;
  }
  CUtensorMap mw2 = mw, my2 = my;
  if (ds) {
    if (int rc = tmap_kmajor_bf16(&mw2, ds->w, d.in_c, d.out_c, block_n / 2, who, "downsample weights")) return rc;
    if (int rc = tmap_nhwc_bf16(&my2, ds->y, d.batch, d.out_h, d.out_w, d.out_c, T2_BOX_W, T2_BOX_H, 1, who, "downsample output")) return rc;
  }
  ConvTc2Args a;
  a.scale = scale; a.bias = bias;
  a.residual = static_cast<const __nv_bfloat16*>(residual);
  a.y = static_cast<__nv_bfloat16*>(y);
  a.B = d.batch; a.Ho = d.out_h; a.Wo = d.out_w; a.Cout = d.out_c;
  a.Cin = d.in_c; a.kh = d.kh; a.kw = d.kw; a.stride = d.stride; a.pad = d.pad; a.dil = d.dil; a.relu = d.relu;
  a.tiles_x = ceil_div(d.out_w, T2_BOX_W);
  a.tiles_per_img = a.tiles_x * ceil_div(d.out_h, T2_BOX_H);
  const long long boxes = (long long)a.tiles_per_img * d.batch;
  HK_REQUIRE(boxes < 0x3fffffffLL, "conv(tcgen05,2cta): too many tiles");
  a.num_boxes = (int)boxes;
  a.num_m_tiles = (a.num_boxes + 3) / 4;
  a.num_n_tiles = d.out_c / block_n;
  a.cblocks = d.in_c / 64;
  a.scale2 = ds ? ds->scale : scale;
  a.bias2 = ds ? ds->bias : bias;
  a.relu2 = ds ? ds->relu : 0;
  // K-block order of the kernel this conv would run on by itself (conv_tc2h accumulates tap column by tap column)
  a.s_major = ds && conv_tc2h_applicable(d);
  { const char* e = getenv("HK_DS_EARLY"); a.early_release = !(e && e[0] == '0'); }   // A/B switch of the block-entry epilogue
#ifdef HK_DIAG
  a.dbg = g_tc2_dbg;
  { const char* m = getenv("HK_TC2_DEBUG"); a.dbg_mode = m ? atoi(m) : 0; }
#endif
  a.bn_acc = static_cast<BnAcc*>(bn_acc);
  a.head_w = head ? head->w : nullptr;
  a.head_b = head ? head->b : nullptr;
  a.head_logits = head ? head->logits : nullptr;
  a.head_k = head ? head->K : 0;
  if (head) return launch_tc2<256, false, false, true>(mx, mw, my, mres, mw2, my2, a, s);
  if (ds) return block_n == 256 ? launch_tc2<256, true, false>(mx, mw, my, mres, mw2, my2, a, s) : launch_tc2<128, true, false>(mx, mw, my, mres, mw2, my2, a, s);
  if (bn_acc) return block_n == 256 ? launch_tc2<256, false, true>(mx, mw, my, mres, mw2, my2, a, s) : launch_tc2<128, false, true>(mx, mw, my, mres, mw2, my2, a, s);
  return block_n == 256 ? launch_tc2<256, false, false>(mx, mw, my, mres, mw2, my2, a, s) : launch_tc2<128, false, false>(mx, mw, my, mres, mw2, my2, a, s);
}

int conv_tc2_launch(const HkConvDesc& d, const void* x, const void* w, const float* scale, const float* bias,
                    const void* residual, void* y, void* bn_acc, cudaStream_t s) {
  return conv_tc2_launch_impl(d, x, w, scale, bias, residual, y, nullptr, bn_acc, s);
}

}  // namespace hk

// Block entry of a stride/channel-changing BasicBlock: y = relu?(scale*conv_kxk(x)+bias), y_ds = scale_ds*conv_1x1(x)+bias_ds in one launch.
extern "C" int hk_conv_ds_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale, const float* bias, void* y,
                              const void* w_ds_packed, const float* scale_ds, const float* bias_ds, void* y_ds, void* stream) {
  using namespace hk;
  HK_REQUIRE(desc && x && w_packed && scale && bias && y && w_ds_packed && scale_ds && bias_ds && y_ds, "hk_conv_ds_fwd: null pointer");
  const HkConvDesc& d = *desc;
  HK_REQUIRE(d.algo == HK_CONV_TCGEN05 && d.in_dtype == HK_BF16 && d.out_dtype == HK_BF16 && !d.in_is_nchw,
             "hk_conv_ds_fwd: tcgen05 path only (NHWC bf16 in and out)");
  HK_REQUIRE(d.batch > 0 && d.in_h > 0 && d.in_w > 0 && d.kh == d.kw && (d.kh & 1) && d.dil > 0 && (d.stride == 1 || d.stride == 2),
             "hk_conv_ds_fwd: bad descriptor");
  HK_REQUIRE(d.pad == d.dil * (d.kh / 2), "hk_conv_ds_fwd: pad must equal dil*(k/2) (the 1x1 conv is the centre tap of the kxk one)");
  HK_REQUIRE(d.out_h == (d.in_h - 1) / d.stride + 1 && d.out_w == (d.in_w - 1) / d.stride + 1, "hk_conv_ds_fwd: out_h/out_w inconsistent");
  HK_REQUIRE(d.out_c % 128 == 0 && d.in_c % 64 == 0, "hk_conv_ds_fwd: needs out_c %% 128 == 0 and in_c %% 64 == 0");
  HK_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w_packed) | reinterpret_cast<uintptr_t>(y) |
               reinterpret_cast<uintptr_t>(w_ds_packed) | reinterpret_cast<uintptr_t>(y_ds)) & 15) == 0,
             "hk_conv_ds_fwd: buffers must be 16-byte aligned");
  HK_REQUIRE(y != y_ds && x != y && x != y_ds, "hk_conv_ds_fwd: buffers must not alias");
  ConvTc2Ds ds{w_ds_packed, scale_ds, bias_ds, y_ds, 0};
  return conv_tc2_launch_impl(d, x, w_packed, scale, bias, nullptr, y, &ds, nullptr, as_stream(stream));
}

// Last conv of the network fused with the K live rows of the scoring conv (see the header): logits += fc_w[:, n-tile] . relu(scale*conv(x)
// + bias + residual) per pixel.  logits (B, K, out_h, out_w) fp32 must be ZERO on entry (two N tiles add into every element).
extern "C" int hk_conv_head_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale, const float* bias,
                                const void* residual_or_null, const float* w_fc, const float* b_fc, int K, float* logits, void* stream) {
  using namespace hk;
  HK_REQUIRE(desc && x && w_packed && scale && bias && w_fc && b_fc && logits, "hk_conv_head_fwd: null pointer");
  const HkConvDesc& d = *desc;
  HK_REQUIRE(d.algo == HK_CONV_TCGEN05 && d.in_dtype == HK_BF16 && d.out_dtype == HK_BF16 && !d.in_is_nchw,
             "hk_conv_head_fwd: tcgen05 path only (NHWC bf16 activations)");
  HK_REQUIRE(d.batch > 0 && d.in_h > 0 && d.in_w > 0 && d.kh > 0 && d.kw > 0 && d.dil > 0 && d.pad >= 0 && d.stride == 1, "hk_conv_head_fwd: bad descriptor");
  const int eh = d.dil * (d.kh - 1) + 1, ew = d.dil * (d.kw - 1) + 1;
  HK_REQUIRE(d.out_h == d.in_h + 2 * d.pad - eh + 1 && d.out_w == d.in_w + 2 * d.pad - ew + 1, "hk_conv_head_fwd: out_h/out_w inconsistent");
  HK_REQUIRE(d.out_c == 512 && d.in_c % 64 == 0, "hk_conv_head_fwd: needs out_c == 512 (two 256-column tiles) and in_c %% 64 == 0");
  HK_REQUIRE(K >= 1 && K <= T2_HEAD_MAX_K, "hk_conv_head_fwd: K=%d outside 1..%d (use hk_conv_bn_act_fwd + hk_head_fwd)", K, T2_HEAD_MAX_K);
  HK_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w_packed) | reinterpret_cast<uintptr_t>(residual_or_null)) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(w_fc) & 15) == 0,
             "hk_conv_head_fwd: buffers must be 16-byte aligned");
  ConvTc2Head head{w_fc, b_fc, logits, K};
  // (the output tensor map is built over the residual / input buffer: HEAD kernels never store through it)
  return conv_tc2_launch_impl(d, x, w_packed, scale, bias, residual_or_null, const_cast<void*>(residual_or_null ? residual_or_null : x), nullptr, nullptr,
                              as_stream(stream), &head);
}
