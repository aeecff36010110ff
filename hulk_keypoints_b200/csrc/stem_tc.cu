// tcgen05 stem: conv 7x7 stride 2 pad 3 (3 -> 64) + folded BN + ReLU  (SURVEY.md k1), bf16 operands, fp32 accumulate,
// and its weight gradient.
//
// Replaces nn.Conv2d(3,64,7,2,3) -> BatchNorm2d -> ReLU of reference src/resnet.py:137-139,199-201 in the bf16
// inference mode (and autograd's weight gradient of that conv under train.py:35).  Cin = 3 is too thin for a TMA
// im2col, so the CTA builds the im2col tile itself:
//   1. the input patch that feeds an 8x16 tile of stem outputs (21 rows x 38 cols x 3 ch; fp32 NCHW, or uint8 HWC) is
//      loaded with coalesced reads one tile ahead into registers, rounded to bf16 and stored pixel-major in shared
//      memory with FOUR channels per pixel (the fourth is zero): one pixel = 8 bytes;
//   2. for one output pixel and one filter row r the 7 taps x 3 channels are then 8 px x 4 ch = 32 contiguous bf16 =
//      64 bytes starting on a 16-byte boundary (2*px pixels in), so an im2col row segment is FOUR 16-byte chunks copied
//      verbatim (LDS.128 -> STS.128, conflict-free) into the 128-byte-swizzled K-major layout tcgen05 expects;
//      K = 7 * 32 = 224, padded to 256 = four 64-wide K blocks.  The eighth pixel / fourth channel of a segment meet
//      zero weights.  (The previous layout, 24 bf16 per filter row with 12 LDS.32 + repacking per segment and per-element
//      index arithmetic in the loads, made the kernel instruction-issue-bound: 1.6k instructions per warp per tile.)
//   3. one thread issues 16 tcgen05.mma (M=128, N=64, K=16) against the weights (64 x 256 bf16, TMA-loaded once per
//      CTA), accumulator in TMEM;
//   4. all 8 warps read TMEM, apply scale/bias(/ReLU) from shared memory and write the bf16 tile into the first K block
//      of the (now idle) A tile, from where one TMA store writes it out.
// Two CTAs per SM (~104 KB smem each) overlap one CTA's global loads/stores with the other's build/MMA.
#include <cuda.h>

#include "hk_common.cuh"
#include "hk_ptx.cuh"

namespace hk {

constexpr int ST_TILE_H = 8, ST_TILE_W = 16;            // stem-output pixels per tile (128 = UMMA M)
constexpr int ST_PATCH_H = 2 * ST_TILE_H + 5;           // 21 input rows
constexpr int ST_PATCH_W = 2 * ST_TILE_W + 6;           // 38 columns (37 used + 1 so 8-pixel segment reads stay in range)
constexpr int ST_PCH = 4;                               // bf16 per patch pixel: 3 channels + one zero
constexpr int ST_SEG = 32;                              // bf16 per filter row in the A tile: 8 px x 4 ch (7 x 3 real taps)
constexpr int ST_K = 256;                               // 7*32 = 224 padded to 4 K blocks of 64
constexpr int ST_KBLOCKS = ST_K / 64;
constexpr int ST_COUT = 64;
constexpr int ST_THREADS = 256;
constexpr int ST_A_BYTES = 128 * 128 * ST_KBLOCKS;      // 64 KB; K block 0 doubles as the output staging tile
constexpr int ST_B_BYTES = ST_COUT * 128 * ST_KBLOCKS;  // 32 KB
constexpr int ST_PATCH_BYTES = (ST_PATCH_H * ST_PATCH_W * ST_PCH * 2 + 15) & ~15;
constexpr int ST_TAIL_BYTES = 64 + 2 * ST_COUT * 4;     // barriers + TMEM pointer, scale[64], bias[64]
constexpr int ST_SMEM_BYTES = 1024 + ST_A_BYTES + ST_B_BYTES + ST_PATCH_BYTES + ST_TAIL_BYTES;
constexpr int ST_ROW_SLOTS = 3;                         // patch rows per warp: w, w+8, w+16 (< 21)

struct StemTcArgs {
  const void* x;    // (B,3,H,W) fp32 NCHW, or (B,H,W,3) uint8 (cv2 layout) in the U8 instantiation
  const float* scale;
  const float* bias;
  __nv_bfloat16* y;  // (B,Ho,Wo,64) bf16
  int B, H, W, Ho, Wo;
  int tiles_x, tiles_per_img, num_tiles;
  int relu;         // 1: ReLU in the epilogue (inference / folded BN); 0: raw affine output (train-mode BN follows)
#ifdef HK_DIAG
  long long* dbg;  // optional phase timeline of CTA 0 (tools/diag_stem_timeline.py); diagnostics build only
#endif
};
#ifdef HK_DIAG
#define ST_DBG(a) ((a).dbg)
#else
#define ST_DBG(a) (static_cast<long long*>(nullptr))
#endif
constexpr int ST_DBG_FIRST = 36;  // first tile (of CTA 0) recorded in the diagnostic timeline: steady state, L2 full of dirty lines
#define ST_STAMP(slot)                                                                            \
  do {                                                                                            \
    if (ST_DBG(a) && blockIdx.x == 0 && tid == 0 && dbg_tile >= ST_DBG_FIRST && dbg_tile < ST_DBG_FIRST + 24) ST_DBG(a)[(dbg_tile - ST_DBG_FIRST) * 8 + (slot)] = clock64(); \
  } while (0)

// byte offset of (row, 16-byte chunk) inside one 128-row x 128-byte K block, SWIZZLE_128B
__device__ __forceinline__ uint32_t sw128_off(int row, int chunk) { return (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4); }

// ---- the input patch of one tile: registers <- global (one tile ahead), shared <- registers ----
// Warp w owns patch rows w, w+8, w+16; lane l owns columns l and l+32 (the latter for l < 6).  fp32 NCHW: three coalesced
// channel loads per pixel; uint8 HWC: three byte loads per pixel (a warp covers 96 contiguous bytes), packed in one register.
template <bool U8>
struct StemPatch {
  uint32_t v[ST_ROW_SLOTS][2][U8 ? 1 : 3];
};
__device__ __forceinline__ void stem_tile_origin(int tile, int tiles_per_img, int tiles_x, int& b, int& ty, int& tx) {
  b = tile / tiles_per_img;
  const int rem = tile - b * tiles_per_img;
  ty = rem / tiles_x;
  tx = rem - ty * tiles_x;
}
template <bool U8>
__device__ __forceinline__ void stem_prefetch_patch(StemPatch<U8>& p, const void* x, int H, int W, int b, int ty, int tx, int warp,
                                                    int lane) {
  const int iy0 = 2 * ty * ST_TILE_H - 3, ix0 = 2 * tx * ST_TILE_W - 3 + lane;
  const bool interior = iy0 >= 0 && iy0 + ST_PATCH_H <= H && ix0 - lane >= 0 && ix0 - lane + ST_PATCH_W <= W;  // CTA-uniform
  const bool has_b = lane < ST_PATCH_W - 32;
  if constexpr (U8) {
    const uint8_t* base = static_cast<const uint8_t*>(x) + ((size_t)b * H * W) * 3;
#pragma unroll
    for (int j = 0; j < ST_ROW_SLOTS; ++j) {
      const int py = warp + 8 * j, iy = iy0 + py;
      const bool row_ok = py < ST_PATCH_H && (interior || (iy >= 0 && iy < H));
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int ix = ix0 + 32 * t;
        const bool ok = row_ok && (t == 0 || has_b) && (interior || (ix >= 0 && ix < W));
        uint32_t v = 0;
        if (ok) {
          const uint8_t* q = base + ((size_t)iy * W + ix) * 3;
          v = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16);
        }
        p.v[j][t][0] = v;
      }
    }
  } else {
    const size_t HW = (size_t)H * W;
    const float* base = static_cast<const float*>(x) + (size_t)b * 3 * HW;
    if (interior) {  // CTA-uniform fast path (all but the border tiles): no per-element bounds logic, strength-reduced addresses
      const float* q0 = base + (size_t)(iy0 + warp) * W + ix0;
#pragma unroll
      for (int j = 0; j < ST_ROW_SLOTS; ++j) {
        const float* q = q0 + (size_t)(8 * j) * W;
        const bool row_ok = warp + 8 * j < ST_PATCH_H;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          p.v[j][0][c] = row_ok ? __float_as_uint(__ldg(q + c * HW)) : 0u;
          p.v[j][1][c] = (row_ok && has_b) ? __float_as_uint(__ldg(q + c * HW + 32)) : 0u;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < ST_ROW_SLOTS; ++j) {
        const int py = warp + 8 * j, iy = iy0 + py;
        const bool row_ok = py < ST_PATCH_H && iy >= 0 && iy < H;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const int ix = ix0 + 32 * t;
          const bool ok = row_ok && (t == 0 || has_b) && ix >= 0 && ix < W;
          const float* q = base + (size_t)(ok ? iy : 0) * W + (ok ? ix : 0);
#pragma unroll
          for (int c = 0; c < 3; ++c) p.v[j][t][c] = ok ? __float_as_uint(__ldg(q + c * HW)) : 0u;
        }
      }
    }
  }
}
template <bool U8>
__device__ __forceinline__ void stem_store_patch(const StemPatch<U8>& p, __nv_bfloat16* patch, int warp, int lane) {
#pragma unroll
  for (int j = 0; j < ST_ROW_SLOTS; ++j) {
    const int py = warp + 8 * j;
    if (py < ST_PATCH_H) {
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        if (t == 0 || lane < ST_PATCH_W - 32) {
          float f0, f1, f2;
          if constexpr (U8) {
            // ToTensor semantics (reference dataset.py:16): bf16_rn(uint8 / 255) == bf16_rn(uint8 * kInv255) for all 256 values (hk_common.cuh)
            const uint32_t v = p.v[j][t][0];
            f0 = (float)(v & 0xffu) * kInv255;
            f1 = (float)((v >> 8) & 0xffu) * kInv255;
            f2 = (float)((v >> 16) & 0xffu) * kInv255;
          } else {
            f0 = __uint_as_float(p.v[j][t][0]);
            f1 = __uint_as_float(p.v[j][t][1]);
            f2 = __uint_as_float(p.v[j][t][2]);
          }
          *reinterpret_cast<uint2*>(patch + (py * ST_PATCH_W + lane + 32 * t) * ST_PCH) = make_uint2(pack_bf16x2(f0, f1), pack_bf16x2(f2, 0.f));
        }
      }
    }
  }
}
// im2col rows into the swizzled A tile: 128 pixels x 7 filter rows = 896 segments of 32 bf16 = four 16-byte chunks each;
// filter row r occupies chunks 4r .. 4r+3 along K, i.e. K block r/2, chunks 4*(r&1) .. +3
__device__ __forceinline__ void stem_build_im2col(const __nv_bfloat16* patch, uint8_t* sA, int tid) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int sidx = tid + i * ST_THREADS;
    if (sidx < 128 * 7) {
      const int row = sidx & 127, r = sidx >> 7;
      const int py = row >> 4, px = row & 15;
      const uint4* src = reinterpret_cast<const uint4*>(patch + ((2 * py + r) * ST_PATCH_W + 2 * px) * ST_PCH);
      const uint4 v0 = src[0], v1 = src[1], v2 = src[2], v3 = src[3];
      uint8_t* blk = sA + (r >> 1) * 16384 + row * 128;
      const int c0 = (r & 1) * 4, sw = row & 7;
      *reinterpret_cast<uint4*>(blk + (((c0 + 0) ^ sw) << 4)) = v0;
      *reinterpret_cast<uint4*>(blk + (((c0 + 1) ^ sw) << 4)) = v1;
      *reinterpret_cast<uint4*>(blk + (((c0 + 2) ^ sw) << 4)) = v2;
      *reinterpret_cast<uint4*>(blk + (((c0 + 3) ^ sw) << 4)) = v3;
    }
  }
}
// k in [224,256) = chunks 4..7 of K block 3 never receive data: zero them once (they meet zero weights, but must be finite)
// (the patch buffer needs no initialisation: all 21 x 38 pixels are rewritten for every tile, zeros outside the image)
__device__ __forceinline__ void stem_zero_k_padding(uint8_t* sA, int tid) {
  for (int i = tid; i < 128 * 4; i += ST_THREADS) {
    const int row = i >> 2, chunk = 4 + (i & 3);
    *reinterpret_cast<uint4*>(sA + 3 * 16384 + sw128_off(row, chunk)) = make_uint4(0, 0, 0, 0);
  }
}

template <bool U8>
__global__ void __launch_bounds__(ST_THREADS, 2)
stem_tc_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_y, const StemTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;                                   // 4 K blocks x [128 rows][128 B]
  uint8_t* sB = smem + ST_A_BYTES;                      // 4 K blocks x [64 rows][128 B]
  uint8_t* sOut = sA;                                   // [128 rows][128 B]: the epilogue reuses K block 0 once the MMAs are done
  __nv_bfloat16* patch = reinterpret_cast<__nv_bfloat16*>(sB + ST_B_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(patch) + ST_PATCH_BYTES);
  uint64_t* w_bar = bars;       // weights landed
  uint64_t* mma_bar = bars + 1; // accumulator ready / A tile free
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2);
  float* s_scale = reinterpret_cast<float*>(bars + 8);  // 64 bytes in: 16-byte aligned
  float* s_bias = s_scale + ST_COUT;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);  // same value, provably warp-uniform for the compiler

  if (tid == 0) {
    ptx::prefetch_tensormap(&map_w);
    ptx::prefetch_tensormap(&map_y);
    ptx::mbar_init(w_bar, 1);
    ptx::mbar_init(mma_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_ptr_smem, 64);
    ptx::tmem_relinquish();
  }
  if (tid >= 64 && tid < 64 + ST_COUT) { s_scale[tid - 64] = a.scale[tid - 64]; s_bias[tid - 64] = a.bias[tid - 64]; }
  stem_zero_k_padding(sA, tid);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (tid == 0) {  // weights: four (64 k x 64 cout) boxes, once per CTA
    ptx::mbar_arrive_expect_tx(w_bar, ST_B_BYTES);
    for (int kb = 0; kb < ST_KBLOCKS; ++kb) ptx::tma_load_2d(sB + kb * 8192, &map_w, w_bar, kb * 64, 0);
  }

  constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, ST_COUT);
  uint32_t mma_phase = 0;
  bool first = true;

  // Software pipeline: the NEXT tile's input patch is fetched into registers while the current tile is built, multiplied and stored.
  StemPatch<U8> pre;
  int b, ty, tx;
  if ((int)blockIdx.x < a.num_tiles) {
    stem_tile_origin(blockIdx.x, a.tiles_per_img, a.tiles_x, b, ty, tx);
    stem_prefetch_patch<U8>(pre, a.x, a.H, a.W, b, ty, tx, warp_u, lane);
  }

  int dbg_tile = 0;
  if (ST_DBG(a) && tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) ST_DBG(a)[192 + (blockIdx.x ? 4 : 0)] = clock64();
  for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++dbg_tile) {
    ST_STAMP(0);
    const int oy0 = ty * ST_TILE_H, ox0 = tx * ST_TILE_W, ob = b;

    // ---- 1. prefetched input patch -> smem, bf16, [y][x][4] ----
    stem_store_patch<U8>(pre, patch, warp_u, lane);
    if (tid == 0) ptx::bulk_wait_group_read0();  // previous tile's TMA store has drained the staging buffer (= K block 0 of sA)
    ST_STAMP(1);
    __syncthreads();  // patch complete; staging free; previous tile's epilogue has drained TMEM (all warps passed it)
    ST_STAMP(2);

    // ---- 2. im2col rows into the swizzled A tile ----
    stem_build_im2col(patch, sA, tid);
    ST_STAMP(3);
    ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to tcgen05
    ptx::tc_fence_before();
    __syncthreads();
    ST_STAMP(4);

    // ---- 3. MMA ----
    if (warp_u == 0 && ptx::elect_one_sync()) {  // warp-uniform branch: descriptors stay in uniform registers
      ptx::tc_fence_after();
      if (first) ptx::mbar_wait(w_bar, 0, 11);
      const uint32_t a0 = ptx::smem_u32(sA), b0 = ptx::smem_u32(sB);
#pragma unroll
      for (int kb = 0; kb < ST_KBLOCKS; ++kb) {
        const uint64_t adesc = ptx::make_smem_desc_sw128(a0 + kb * 16384);
        const uint64_t bdesc = ptx::make_smem_desc_sw128(b0 + kb * 8192);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (kb * 64 + k * 16 < 7 * ST_SEG)  // k >= 224 is zero padding on both operands: those two K steps are skipped
            ptx::umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
      }
      ptx::umma_commit(mma_bar);
    }
    first = false;
    // next tile's input patch -> registers while the tensor core works on this one
    if (tile + (int)gridDim.x < a.num_tiles) {
      stem_tile_origin(tile + gridDim.x, a.tiles_per_img, a.tiles_x, b, ty, tx);
      stem_prefetch_patch<U8>(pre, a.x, a.H, a.W, b, ty, tx, warp_u, lane);
    }
    ST_STAMP(5);

    // ---- 4. epilogue (all 8 warps: warp%4 = TMEM lane quarter, warp/4 = channel half) ----
    ptx::mbar_wait(mma_bar, mma_phase, 12);
    mma_phase ^= 1;
    ptx::tc_fence_after();
    ST_STAMP(6);
    {
      const int q = warp & 3, c0 = (warp >> 2) * 32;
      const int row = q * 32 + lane;
      uint8_t* my_row = sOut + row * 128;
      const int sw = row & 7;
      uint32_t r[32];
      ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c0, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int c = c0 + g * 8;
        const float4 s0 = *reinterpret_cast<const float4*>(s_scale + c);
        const float4 s1 = *reinterpret_cast<const float4*>(s_scale + c + 4);
        const float4 t0 = *reinterpret_cast<const float4*>(s_bias + c);
        const float4 t1 = *reinterpret_cast<const float4*>(s_bias + c + 4);
        const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float bi[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[j] = fmaf(__uint_as_float(r[g * 8 + j]), sc[j], bi[j]);
          if (a.relu) v[j] = fmaxf(v[j], 0.f);
        }
        *reinterpret_cast<uint4*>(my_row + ((((c >> 3) ^ sw) & 7) << 4)) =
            make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      }
      ptx::tc_fence_before();
      ptx::fence_proxy_async_smem();
    }
    __syncthreads();
    if (tid == 0) {  // one coalesced tile store; rows / columns beyond the image are clipped by the TMA unit
      ptx::tma_store_4d(&map_y, sOut, 0, ox0, oy0, ob);
      ptx::bulk_commit_group();
    }
    ST_STAMP(7);
  }

  if (ST_DBG(a) && tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) ST_DBG(a)[193 + (blockIdx.x ? 4 : 0)] = clock64();
  if (tid == 0) ptx::bulk_wait_group0();
  if (ST_DBG(a) && tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) {
    ST_DBG(a)[194 + (blockIdx.x ? 4 : 0)] = clock64();
    ST_DBG(a)[195 + (blockIdx.x ? 4 : 0)] = dbg_tile;
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 64);
  }
}

// ------------------------------------------------------------------------------------------------ stem weight gradient
// dW[co][c][r][s] = sum_{b,oy,ox} dY[b,oy,ox,co] * X[b,c,2oy-3+r,2ox-3+s]   (autograd of the stem conv, reference
// src/resnet.py:137 under train.py:35), as a tcgen05 GEMM whose reduction runs over the output pixels:
//   D[M = co (64, duplicated to 128), N = k (256)] += dY_tile^T[co, 128 px] * im2col_tile[128 px, k]
// The im2col tile is built exactly like the forward kernel's A tile ([128 px][256 k], 128-byte-swizzled); here it is the
// B operand read MN-major (k contiguous, pixels = GEMM-K strided: 8-pixel groups 1024 B apart, 64-wide k groups 16 KB apart).
// The dY tile (128 px x 64 co bf16) is one SWIZZLE_128B TMA box, loaded twice so the A operand has 128 rows (rows 64..127 of
// the accumulator repeat rows 0..63 and are never read).  The fp32 accumulator (128 lanes x 256 columns of TMEM) lives across
// ALL tiles of the persistent CTA; one epilogue at the end writes the CTA's partial [64 co][256 k], summed in a fixed order by
// stem_wgrad_tc_finalize_kernel (deterministic, no atomics).  x is rounded to bf16 exactly as in the forward kernel.
constexpr int SWG_DY_TILE_BYTES = 128 * 128;                           // 128 px x 64 co bf16
constexpr int SWG_DY_BYTES = 2 * SWG_DY_TILE_BYTES;                     // two copies: accumulator rows 0..63 and 64..127
constexpr int SWG_SMEM_BYTES = 1024 + ST_A_BYTES + SWG_DY_BYTES + ST_PATCH_BYTES + 64;
constexpr int SWG_TMEM_COLS = 256;

struct StemWgradArgs {
  const float* x;     // (B,3,H,W) fp32 NCHW
  float* partial;     // [grid][64 co][256 k] fp32
  int B, H, W, Ho, Wo;
  int tiles_x, tiles_per_img, num_tiles;
};

// MN-major SWIZZLE_128B operand made of [128 px][128 B] blocks: LBO = 16 KB between 64-element groups along M/N,
// SBO = 1024 B between 8-pixel groups along K
__device__ __forceinline__ uint64_t make_smem_desc_mn_sw128_16k(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(16384 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__global__ void __launch_bounds__(ST_THREADS, 2)
stem_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy, const StemWgradArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;                                   // im2col: 4 k blocks x [128 px][128 B]
  uint8_t* sDy = smem + ST_A_BYTES;                     // 2 x [128 px][128 B]
  __nv_bfloat16* patch = reinterpret_cast<__nv_bfloat16*>(sDy + SWG_DY_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(patch) + ST_PATCH_BYTES);
  uint64_t* dy_bar = bars;       // dY tile landed
  uint64_t* mma_bar = bars + 1;  // this tile's MMAs done: sA / sDy may be overwritten
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);

  if (tid == 0) {
    ptx::prefetch_tensormap(&map_dy);
    ptx::mbar_init(dy_bar, 1);
    ptx::mbar_init(mma_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_ptr_smem, SWG_TMEM_COLS);
    ptx::tmem_relinquish();
  }
  stem_zero_k_padding(sA, tid);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, ST_K) | (1u << 15) | (1u << 16);  // A and B MN-major
  uint32_t phase = 0;   // parity of dy_bar / mma_bar for the current tile (each completes once per tile)
  bool first = true;

  StemPatch<false> pre;
  int b, ty, tx;
  if ((int)blockIdx.x < a.num_tiles) {
    stem_tile_origin(blockIdx.x, a.tiles_per_img, a.tiles_x, b, ty, tx);
    stem_prefetch_patch<false>(pre, a.x, a.H, a.W, b, ty, tx, warp_u, lane);
  }

  for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
    const int oy0 = ty * ST_TILE_H, ox0 = tx * ST_TILE_W, ob = b;

    // ---- 1. prefetched input patch -> smem (the patch buffer is not an MMA operand) ----
    stem_store_patch<false>(pre, patch, warp_u, lane);
    // ---- 2. previous tile's MMAs have finished reading sA / sDy; fetch this tile's dY ----
    if (!first) ptx::mbar_wait(mma_bar, phase ^ 1, 14);
    if (tid == 0) {
      ptx::mbar_arrive_expect_tx(dy_bar, SWG_DY_BYTES);
      ptx::tma_load_4d(sDy, &map_dy, dy_bar, 0, ox0, oy0, ob);                      // pixels beyond the image arrive as zeros
      ptx::tma_load_4d(sDy + SWG_DY_TILE_BYTES, &map_dy, dy_bar, 0, ox0, oy0, ob);
    }
    __syncthreads();  // patch complete

    // ---- 3. im2col rows into the swizzled tile (same layout as the forward kernel's A tile) ----
    stem_build_im2col(patch, sA, tid);
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before();
    __syncthreads();

    // ---- 4. MMA: 8 steps of 16 pixels ----
    if (warp_u == 0) {
      ptx::mbar_wait(dy_bar, phase, 15);
      ptx::tc_fence_after();
      if (ptx::elect_one_sync()) {
        const uint64_t adesc = make_smem_desc_mn_sw128_16k(ptx::smem_u32(sDy));
        const uint64_t bdesc = make_smem_desc_mn_sw128_16k(ptx::smem_u32(sA));
#pragma unroll
        for (int k = 0; k < 8; ++k)  // 16 pixels = 2048 bytes further along the reduction: +128 in the (addr >> 4) field
          ptx::umma_bf16(tmem_base, adesc + 128 * k, bdesc + 128 * k, idesc, (!first || k != 0) ? 1u : 0u);
        ptx::umma_commit(mma_bar);
      }
      __syncwarp();
    }
    first = false;
    phase ^= 1;
    if (tile + (int)gridDim.x < a.num_tiles) {
      stem_tile_origin(tile + gridDim.x, a.tiles_per_img, a.tiles_x, b, ty, tx);
      stem_prefetch_patch<false>(pre, a.x, a.H, a.W, b, ty, tx, warp_u, lane);
    }
  }

  // ---- epilogue: the CTA's accumulated [64 co][256 k] -> partial (warp%4 = TMEM lane quarter, warp/4 = column half) ----
  if (!first) {
    ptx::mbar_wait(mma_bar, phase ^ 1, 16);
    ptx::tc_fence_after();
    const int q = warp & 3, c0 = (warp >> 2) * (ST_K / 2);
    if (q < 2) {  // rows 64..127 duplicate rows 0..63
      const int co = q * 32 + lane;
      float* dst = a.partial + ((size_t)blockIdx.x * ST_COUT + co) * ST_K + c0;
#pragma unroll 1
      for (int cc = 0; cc < ST_K / 2; cc += 32) {
        uint32_t r[32];
        ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c0 + cc, r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int g = 0; g < 8; ++g)
          *reinterpret_cast<float4*>(dst + cc + g * 4) = make_float4(__uint_as_float(r[g * 4]), __uint_as_float(r[g * 4 + 1]),
                                                                      __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3]));
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, SWG_TMEM_COLS);
  }
}

// dw (64,3,7,7) OIHW (+)= sum over CTAs of partial[cta][co][r*32 + s*4 + c]; fixed order, double accumulation
__global__ void __launch_bounds__(256) stem_wgrad_tc_finalize_kernel(const float* __restrict__ partial, int nblk, float* __restrict__ dw,
                                                                    int accumulate) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;   // co * 147 + (c*7 + r)*7 + s
  if (j >= 64 * 147) return;
  const int co = j / 147, t = j - co * 147;
  const int c = t / 49, rs = t - c * 49, r = rs / 7, sft = rs - r * 7;
  const float* p = partial + (size_t)co * ST_K + r * ST_SEG + sft * ST_PCH + c;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int b = 0;
  for (; b + 4 <= nblk; b += 4) {
    s0 += (double)p[(size_t)(b + 0) * (ST_COUT * ST_K)];
    s1 += (double)p[(size_t)(b + 1) * (ST_COUT * ST_K)];
    s2 += (double)p[(size_t)(b + 2) * (ST_COUT * ST_K)];
    s3 += (double)p[(size_t)(b + 3) * (ST_COUT * ST_K)];
  }
  for (; b < nblk; ++b) s0 += (double)p[(size_t)b * (ST_COUT * ST_K)];
  dw[j] = (accumulate ? dw[j] : 0.f) + (float)((s0 + s1) + (s2 + s3));
}

// OIHW (64,3,7,7) fp32 -> (64, 256) bf16 with k = r*32 + s*4 + c, zeros elsewhere
__global__ void stem_pack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ST_COUT * ST_K) return;
  const int o = i / ST_K, k = i - o * ST_K;
  const int r = k / ST_SEG, j = k - r * ST_SEG;
  const int s = j / ST_PCH, c = j - s * ST_PCH;
  float v = 0.f;
  if (r < 7 && s < 7 && c < 3) v = w[((o * 3 + c) * 7 + r) * 7 + s];
  out[i] = __float2bfloat16_rn(v);
}

}  // namespace hk

extern "C" {

size_t hk_stem_packed_weight_bytes(void) { return (size_t)hk::ST_COUT * hk::ST_K * sizeof(__nv_bfloat16); }

int hk_stem_pack_weights(const float* w_oihw, void* w_out, void* stream) {
  using namespace hk;
  HK_REQUIRE(w_oihw && w_out, "hk_stem_pack_weights: null pointer");
  stem_pack_kernel<<<ceil_div(ST_COUT * ST_K, 256), 256, 0, as_stream(stream)>>>(w_oihw, static_cast<__nv_bfloat16*>(w_out));
  return check_launch("stem_pack_kernel");
}

#ifdef HK_DIAG
static long long* g_stem_dbg = nullptr;
// Diagnostic hook of the --diag build (not in the public header): device buffer of 24*8 int64 receiving CTA 0's phase clocks.
__attribute__((visibility("default"))) void hk_debug_set_stem_timeline(long long* dev_buf) { g_stem_dbg = dev_buf; }
#endif

static int stem_launch(const void* x, bool u8, const void* w_packed, const float* scale, const float* bias, void* y_nhwc, int B,
                       int H, int W, void* stream, int relu = 1) {
  using namespace hk;
  HK_REQUIRE(x && w_packed && scale && bias && y_nhwc, "hk_stem_fwd: null pointer");
  HK_REQUIRE(B > 0 && H >= 7 && W >= 7, "hk_stem_fwd: bad shape");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(w_packed) & 15) == 0 && (reinterpret_cast<uintptr_t>(y_nhwc) & 15) == 0,
             "hk_stem_fwd: buffers must be 16-byte aligned");
  const int Ho = (H + 6 - 7) / 2 + 1, Wo = (W + 6 - 7) / 2 + 1;
  const char* who = "hk_stem_fwd";
  CUtensorMap mw, my;
  if (int rc = tmap_kmajor_bf16(&mw, w_packed, ST_K, ST_COUT, ST_COUT, who, "weights")) return rc;
  if (int rc = tmap_nhwc_bf16(&my, y_nhwc, B, Ho, Wo, 64, ST_TILE_W, ST_TILE_H, 1, who, "output")) return rc;
  StemTcArgs a;
  a.x = x; a.scale = scale; a.bias = bias; a.y = static_cast<__nv_bfloat16*>(y_nhwc);
  a.B = B; a.H = H; a.W = W;
#ifdef HK_DIAG
  a.dbg = g_stem_dbg;
#endif
  a.relu = relu;
  a.Ho = Ho;
  a.Wo = Wo;
  a.tiles_x = ceil_div(a.Wo, ST_TILE_W);
  a.tiles_per_img = a.tiles_x * ceil_div(a.Ho, ST_TILE_H);
  const long long nt = (long long)a.tiles_per_img * B;
  HK_REQUIRE(nt < 0x7fffffffLL, "hk_stem_fwd: too many tiles");
  a.num_tiles = (int)nt;
  if (int rc = u8 ? opt_in_smem<stem_tc_kernel<true>>(ST_SMEM_BYTES, who) : opt_in_smem<stem_tc_kernel<false>>(ST_SMEM_BYTES, who)) return rc;
  int grid = 2 * sm_count();
  if (grid > a.num_tiles) grid = a.num_tiles;
  if (u8) stem_tc_kernel<true><<<grid, ST_THREADS, ST_SMEM_BYTES, as_stream(stream)>>>(mw, my, a);
  else stem_tc_kernel<false><<<grid, ST_THREADS, ST_SMEM_BYTES, as_stream(stream)>>>(mw, my, a);
  return check_launch("stem_tc_kernel");
}

int hk_stem_fwd(const float* x_nchw, const void* w_packed, const float* scale, const float* bias, void* y_nhwc, int B, int H,
                int W, void* stream) {
  return stem_launch(x_nchw, false, w_packed, scale, bias, y_nhwc, B, H, W, stream);
}

int hk_stem_conv_fwd(const float* x_nchw, const void* w_packed, const float* scale, const float* bias, void* y_nhwc, int B, int H,
                     int W, int relu, void* stream) {
  return stem_launch(x_nchw, false, w_packed, scale, bias, y_nhwc, B, H, W, stream, relu);
}

int hk_stem_fwd_u8(const uint8_t* x_nhwc_u8, const void* w_packed, const float* scale, const float* bias, void* y_nhwc, int B,
                   int H, int W, void* stream) {
  return stem_launch(x_nhwc_u8, true, w_packed, scale, bias, y_nhwc, B, H, W, stream);
}

size_t hk_stem_wgrad_workspace_bytes(void) { return (size_t)hk::sm_count() * 2 * hk::ST_COUT * hk::ST_K * sizeof(float); }

int hk_stem_wgrad(const float* x_nchw, const void* dy_nhwc, float* dw_oihw, int accumulate, int B, int H, int W, void* ws,
                  size_t ws_bytes, void* stream) {
  using namespace hk;
  HK_REQUIRE(x_nchw && dy_nhwc && dw_oihw && ws, "hk_stem_wgrad: null pointer");
  HK_REQUIRE(B > 0 && H >= 7 && W >= 7, "hk_stem_wgrad: bad shape");
  HK_REQUIRE(ws_bytes >= hk_stem_wgrad_workspace_bytes(), "hk_stem_wgrad: workspace too small");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(dy_nhwc) & 15) == 0 && (reinterpret_cast<uintptr_t>(ws) & 15) == 0,
             "hk_stem_wgrad: buffers must be 16-byte aligned");
  const int Ho = (H + 6 - 7) / 2 + 1, Wo = (W + 6 - 7) / 2 + 1;
  CUtensorMap mdy;
  if (int rc = tmap_nhwc_bf16(&mdy, dy_nhwc, B, Ho, Wo, 64, ST_TILE_W, ST_TILE_H, 1, "hk_stem_wgrad", "dy")) return rc;
  StemWgradArgs a;
  a.x = x_nchw; a.partial = static_cast<float*>(ws);
  a.B = B; a.H = H; a.W = W; a.Ho = Ho; a.Wo = Wo;
  a.tiles_x = ceil_div(Wo, ST_TILE_W);
  a.tiles_per_img = a.tiles_x * ceil_div(Ho, ST_TILE_H);
  const long long nt = (long long)a.tiles_per_img * B;
  HK_REQUIRE(nt < 0x7fffffffLL, "hk_stem_wgrad: too many tiles");
  a.num_tiles = (int)nt;
  if (int rc = opt_in_smem<stem_wgrad_tc_kernel>(SWG_SMEM_BYTES, "hk_stem_wgrad")) return rc;
  int grid = 2 * sm_count();
  if (grid > a.num_tiles) grid = a.num_tiles;
  stem_wgrad_tc_kernel<<<grid, ST_THREADS, SWG_SMEM_BYTES, as_stream(stream)>>>(mdy, a);
  int rc = check_launch("stem_wgrad_tc_kernel");
  if (rc) return rc;
  stem_wgrad_tc_finalize_kernel<<<ceil_div(64 * 147, 256), 256, 0, as_stream(stream)>>>(static_cast<const float*>(ws), grid, dw_oihw,
                                                                                       accumulate);
  return check_launch("stem_wgrad_tc_finalize_kernel");
}

}  // extern "C"
