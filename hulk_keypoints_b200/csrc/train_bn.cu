// Train-mode BatchNorm2d (+ residual add, ReLU) forward and backward on NHWC bf16 activations.
//
// Reference: nn.BatchNorm2d in train() mode at src/resnet.py:46,49,139,187 as called from BasicBlock.forward
// (src/resnet.py:53-69) and ResNet.forward (:199-201), with autograd's backward (train.py:35).
//   forward : mu = mean_p y, var = mean_p (y-mu)^2 (biased), xhat = (y-mu)*rsqrt(var+eps),
//             out = relu(gamma*xhat + beta [+ residual]); running stats updated with momentum (unbiased var)
//   backward: d' = dout * [out > 0];  dbeta = sum d';  dgamma = sum d'*xhat;
//             dy = gamma*invstd * (d' - dbeta/N - xhat*dgamma/N)
// All four kernels are HBM-bound streaming passes (16-byte vectors of 8 bf16 channels); the reductions are two-level
// (fixed grid of per-block fp32 partials, then a double-precision finalize) and therefore deterministic -- no atomics.
#include <cooperative_groups.h>

#include "hk_common.cuh"
#include "hk_bn_acc.cuh"

namespace hk {

namespace cg = cooperative_groups;

constexpr int BN_THREADS = 256;
constexpr int BN_MAX_BLOCKS = 592;  // 148 SMs x 4

struct Vec8 {
  float v[8];
};
__device__ __forceinline__ Vec8 load8(const __nv_bfloat16* p) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  Vec8 r;
  unpack_bf16x2(u.x, r.v[0], r.v[1]);
  unpack_bf16x2(u.y, r.v[2], r.v[3]);
  unpack_bf16x2(u.z, r.v[4], r.v[5]);
  unpack_bf16x2(u.w, r.v[6], r.v[7]);
  return r;
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

// Block-level reduction of two per-thread 8-channel accumulators over the row lanes of the block, written as
// partial[blockIdx][0..1][C].  Thread layout: cg = tid % CG (channel group of 8), ty = tid / CG.
template <class Emit>
__device__ __forceinline__ void block_reduce_2x8_emit(const float (&a)[8], const float (&b)[8], int C, Emit emit) {
  __shared__ float sh[2 * BN_THREADS * 8];  // [2][rows][C] with rows*C = 256*8
  const int CG = C >> 3, cg = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float* s0 = sh + (ty * C + cg * 8);
  float* s1 = s0 + BN_THREADS * 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) { s0[j] = a[j]; s1[j] = b[j]; }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += BN_THREADS) {
    const int which = c / C, ch = c - which * C;
    const float* src = sh + which * BN_THREADS * 8 + ch;
    float acc = 0.f;
    for (int r = 0; r < rows; ++r) acc += src[r * C];
    emit(c, acc);
  }
}
__device__ __forceinline__ void block_reduce_2x8(const float (&a)[8], const float (&b)[8], int C, float* __restrict__ partial) {
  __shared__ float sh[2 * BN_THREADS * 8];  // [2][rows][C] with rows*C = 256*8
  const int CG = C >> 3, cg = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float* s0 = sh + (ty * C + cg * 8);
  float* s1 = s0 + BN_THREADS * 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) { s0[j] = a[j]; s1[j] = b[j]; }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += BN_THREADS) {
    const int which = c / C, ch = c - which * C;
    const float* src = sh + which * BN_THREADS * 8 + ch;
    float acc = 0.f;
    for (int r = 0; r < rows; ++r) acc += src[r * C];
    partial[(size_t)blockIdx.x * 2 * C + c] = acc;
  }
}

// ---- forward statistics ----
__global__ void __launch_bounds__(BN_THREADS) bn_stats_partial_kernel(const __nv_bfloat16* __restrict__ y, long long P, int C,
                                                                     float* __restrict__ partial) {
  const int CG = C >> 3, cg = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (long long r = (long long)blockIdx.x * rows + ty; r < P; r += (long long)gridDim.x * rows) {
    const Vec8 v = load8(y + r * C + cg * 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += v.v[j]; q[j] = fmaf(v.v[j], v.v[j], q[j]); }
  }
  block_reduce_2x8(s, q, C, partial);
}

// Finalize kernels: 1024 threads = 32 channels x 32 slices of the per-block partials (coalesced across channels; every thread has
// up to 8 independent loads in flight and walks <= 19 of the 592 partials -- one thread per channel walking them serially cost
// 170 us per launch, 8 slices with 2-deep unrolling still 15 us: the loop is pure L2 latency).  Fixed order => deterministic.
constexpr int BN_FIN_SLICES = 32;
constexpr int BN_FIN_THREADS = 32 * BN_FIN_SLICES;
__device__ __forceinline__ void bn_sum_partials(const float* __restrict__ partial, int nblocks, int C, int c, double& s, double& q) {
  __shared__ double sh[2][BN_FIN_SLICES][33];
  const int lane_c = threadIdx.x & 31, slice = threadIdx.x >> 5;
  float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
  if (c < C) {
    int blk = slice;
    for (; blk + 3 * BN_FIN_SLICES < nblocks; blk += 4 * BN_FIN_SLICES) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        a[u] += partial[(size_t)(blk + u * BN_FIN_SLICES) * 2 * C + c];
        b[u] += partial[(size_t)(blk + u * BN_FIN_SLICES) * 2 * C + C + c];
      }
    }
    for (; blk < nblocks; blk += BN_FIN_SLICES) {
      a[0] += partial[(size_t)blk * 2 * C + c];
      b[0] += partial[(size_t)blk * 2 * C + C + c];
    }
  }
  sh[0][slice][lane_c] = ((double)a[0] + (double)a[1]) + ((double)a[2] + (double)a[3]);
  sh[1][slice][lane_c] = ((double)b[0] + (double)b[1]) + ((double)b[2] + (double)b[3]);
  __syncthreads();
  double s4[4] = {0.0, 0.0, 0.0, 0.0}, q4[4] = {0.0, 0.0, 0.0, 0.0};
  if (threadIdx.x < 32) {
#pragma unroll
    for (int i = 0; i < BN_FIN_SLICES; ++i) { s4[i & 3] += sh[0][i][lane_c]; q4[i & 3] += sh[1][i][lane_c]; }
  }
  s = (s4[0] + s4[1]) + (s4[2] + s4[3]);
  q = (q4[0] + q4[1]) + (q4[2] + q4[3]);
}

// mean / invstd, the fused affine (scale, shift) of the apply pass, running statistics
__global__ void __launch_bounds__(BN_FIN_THREADS) bn_stats_finalize_kernel(const float* __restrict__ partial, int nblocks, long long P, int C, const float* __restrict__ gamma,
                                         const float* __restrict__ beta, float* __restrict__ running_mean,
                                         float* __restrict__ running_var, float momentum, float eps, float* __restrict__ mean_out,
                                         float* __restrict__ invstd_out, float* __restrict__ scale_out, float* __restrict__ shift_out) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  double s, q;
  bn_sum_partials(partial, nblocks, C, c, s, q);
  if (c >= C || threadIdx.x >= 32) return;
  const double n = (double)P;
  const double mean = s / n;
  double var = q / n - mean * mean;
  if (var < 0.0) var = 0.0;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float g = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
  mean_out[c] = (float)mean;
  invstd_out[c] = invstd;
  scale_out[c] = g * invstd;
  shift_out[c] = bt - (float)mean * g * invstd;
  if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
  if (running_var) {
    const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

// ---- forward apply: out = relu?(y*scale + shift [+ residual]) ----
__global__ void __launch_bounds__(BN_THREADS) bn_apply_fwd_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                                                                 const float* __restrict__ shift,
                                                                 const __nv_bfloat16* __restrict__ residual, int relu,
                                                                 __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ relu_bits,
                                                                 long long nvec, int C) {
  // the grid stride (gridDim*256) is a multiple of C/8, so a thread keeps its 8 channels: coefficients live in registers
  const int cg = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) % (C >> 3));
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = __ldg(scale + cg * 8 + j); sh[j] = __ldg(shift + cg * 8 + j); }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    const Vec8 v = load8(y + i * 8);
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(v.v[j], sc[j], sh[j]);
    if (residual) {
      const Vec8 r = load8(residual + i * 8);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] += r.v[j];
    }
    if (relu) {
      if (relu_bits) {  // bit j = [out_j > 0]: the ReLU mask of the backward pass at 1/16 of the bytes of `out`
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) m |= (o[j] > 0.f ? 1u : 0u) << j;
        relu_bits[i] = (uint8_t)m;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fmaxf(o[j], 0.f);
    }
    store8(out + i * 8, o);
  }
}

// ---- backward reduce: s1 = sum d', s2 = sum d'*xhat with d' = dout*[out>0] ----
template <bool BITS>
__global__ void __launch_bounds__(BN_THREADS) bn_bwd_partial_kernel(const __nv_bfloat16* __restrict__ dout,
                                                                   const void* __restrict__ out_mask,
                                                                   const __nv_bfloat16* __restrict__ y, const float* __restrict__ mean,
                                                                   const float* __restrict__ invstd, long long P, int C,
                                                                   float* __restrict__ partial) {
  const int CG = C >> 3, cg = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float mu[8], is[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { mu[j] = mean[cg * 8 + j]; is[j] = invstd[cg * 8 + j]; }
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (long long r = (long long)blockIdx.x * rows + ty; r < P; r += (long long)gridDim.x * rows) {
    const long long off = r * C + cg * 8;
    Vec8 d = load8(dout + off);
    if (out_mask) {
      if constexpr (BITS) {
        const uint32_t m = static_cast<const uint8_t*>(out_mask)[off >> 3];
#pragma unroll
        for (int j = 0; j < 8; ++j) d.v[j] = (m >> j) & 1u ? d.v[j] : 0.f;
      } else {
        const Vec8 m = load8(static_cast<const __nv_bfloat16*>(out_mask) + off);
#pragma unroll
        for (int j = 0; j < 8; ++j) d.v[j] = m.v[j] > 0.f ? d.v[j] : 0.f;
      }
    }
    const Vec8 v = load8(y + off);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s1[j] += d.v[j];
      s2[j] = fmaf(d.v[j], (v.v[j] - mu[j]) * is[j], s2[j]);
    }
  }
  block_reduce_2x8(s1, s2, C, partial);
}

// dgamma, dbeta (fp32 parameter gradients; accumulate != 0 adds to what is there) and the coefficients of the apply pass:
//   coef[0][c] = gamma*invstd, coef[1][c] = dbeta/N, coef[2][c] = dgamma/N
__global__ void __launch_bounds__(BN_FIN_THREADS) bn_bwd_finalize_kernel(const float* __restrict__ partial, int nblocks, long long P, int C, const float* __restrict__ gamma,
                                       const float* __restrict__ invstd, float* __restrict__ dgamma, float* __restrict__ dbeta,
                                       int accumulate, float* __restrict__ coef) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  double s1, s2;
  bn_sum_partials(partial, nblocks, C, c, s1, s2);
  if (c >= C || threadIdx.x >= 32) return;
  const float g = gamma ? gamma[c] : 1.f;
  if (dbeta) dbeta[c] = (accumulate ? dbeta[c] : 0.f) + (float)s1;
  if (dgamma) dgamma[c] = (accumulate ? dgamma[c] : 0.f) + (float)s2;
  coef[c] = g * invstd[c];
  coef[C + c] = (float)(s1 / (double)P);
  coef[2 * C + c] = (float)(s2 / (double)P);
}

// dy = coef0 * (d' - coef1 - xhat*coef2) = k0*d' + k1*y + k2 per channel; optionally also writes d' (the gradient that flows
// into the shortcut branch).  The thread's 8 channels are loop-invariant (see bn_apply_fwd_kernel): 24 coefficients in registers.
template <bool BITS>
__global__ void __launch_bounds__(BN_THREADS) bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dout,
                                                                 const void* __restrict__ out_mask,
                                                                 const __nv_bfloat16* __restrict__ y, const float* __restrict__ mean,
                                                                 const float* __restrict__ invstd, const float* __restrict__ coef,
                                                                 __nv_bfloat16* __restrict__ dy, __nv_bfloat16* __restrict__ dmasked,
                                                                 long long nvec, int C) {
  const int c0 = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) % (C >> 3)) * 8;
  float k0[8], k1[8], k2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = c0 + j;
    const float a = __ldg(coef + c), is = __ldg(invstd + c), mu = __ldg(mean + c);
    k0[j] = a;
    k1[j] = -a * __ldg(coef + 2 * C + c) * is;
    k2[j] = -a * __ldg(coef + C + c) - k1[j] * mu;
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    Vec8 d = load8(dout + i * 8);
    if (out_mask) {
      if constexpr (BITS) {
        const uint32_t m = static_cast<const uint8_t*>(out_mask)[i];
#pragma unroll
        for (int j = 0; j < 8; ++j) d.v[j] = (m >> j) & 1u ? d.v[j] : 0.f;
      } else {
        const Vec8 m = load8(static_cast<const __nv_bfloat16*>(out_mask) + i * 8);
#pragma unroll
        for (int j = 0; j < 8; ++j) d.v[j] = m.v[j] > 0.f ? d.v[j] : 0.f;
      }
    }
    if (dmasked) store8(dmasked + i * 8, d.v);
    const Vec8 v = load8(y + i * 8);
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(k0[j], d.v[j], fmaf(k1[j], v.v[j], k2[j]));
    store8(dy + i * 8, o);
  }
}


// ================================================================================================================================
// Accumulator variant (the training engine's path): the per-block partial sums go straight into per-channel 128-bit FIXED-POINT
// accumulators with integer atomics.  Integer addition is associative, so the totals are exact sums of the fp32 block partials
// whatever order the blocks retire in: deterministic like the two-level reduction above, but without the [blocks][2][C] scratch
// and -- the point -- without a finalize launch: the apply kernels turn the accumulators into their per-channel coefficients in
// their own prologue (each block: C channels over 256 threads; block 0 also writes the saved statistics / running stats /
// parameter gradients).  BatchNorm forward = 2 launches instead of 3, backward = 2 instead of 3 (72 launches per train step).
// Accumulators must be zero when the reduce kernel starts (the engine clears all of them with one memset node per graph).
constexpr int BN_ACC_MAX_C = 2048;

// Reduce kernels run as clusters of 8 CTAs: every CTA leaves its 2*C block sums in shared memory, CTA 0 of the cluster adds the eight
// of them over DSMEM in rank order (fixed order: deterministic) and issues the atomics -- 1/8 of the atomic traffic of a per-CTA scheme
// (at C = 512 and 592 blocks that was 1.2 M same-address L2 atomics per launch, ~8 us; now ~71 clusters x 2 K).
constexpr int BN_CLUSTER = 8;
constexpr int BN_ACC_MAX_BLOCKS = 1184;   // upper bound only (148 SMs x 8 blocks); the grid is one resident wave of clusters, see bn_grid_acc_rows

// Tunables of the accumulator kernels (tools/diag_bn_kernels.py + tools/build_bn_variants.sh; DESIGN 3.5).  These kernels are pure streams:
// their throughput is the bytes they keep in flight (resident threads x independent 16-byte loads per thread), not their arithmetic --
// *_U = rows / vectors a thread has in flight, *_MINB = resident blocks per SM the register allocation is held to, *_CONTIG = 1: the
// U pieces of a thread are neighbours (a block reads U contiguous 4 KB pieces of every operand per iteration), 0: one grid stride apart.
#ifndef BN_STATS_U
#define BN_STATS_U 4
#endif
#ifndef BN_BWDRED_U
#define BN_BWDRED_U 2
#endif
#ifndef BN_RED_MINB
#define BN_RED_MINB 4
#endif
#ifndef BN_RED_CONTIG
#define BN_RED_CONTIG 1
#endif
#ifndef BN_APPLY_U
#define BN_APPLY_U 4
#endif
#ifndef BN_APPLY_MINB
#define BN_APPLY_MINB 3
#endif
#ifndef BN_APPLY_CONTIG
#define BN_APPLY_CONTIG 1
#endif
// least chunks (U rows x 256/(C/8) rows) per reduce block.  Small-batch launches want MANY blocks: fatter blocks (8 / 16 / 32 chunks, and
// likewise 4 / 8 / 16 per apply block) made the batch-4 train step 3 % / 12 % / 31 % slower -- parallelism beats the per-block emit /
// coefficient prologue
#ifndef BN_RED_MIN_CHUNKS
#define BN_RED_MIN_CHUNKS 4
#endif

// Shared-memory footprints are kept small on purpose (dynamic, sized by C): these kernels share the SMs with the weight-gradient
// kernels of the second stream (one 198 KB CTA per SM), and a BatchNorm block that does not fit next to one simply waits for it.
// Block sums of two per-thread 8-channel accumulators through ONE 8 KB buffer (a, then b): half the static shared memory of
// block_reduce_2x8, so that more reduce blocks fit beside a weight-gradient CTA.  Same per-channel summation order (rows ascending).
__device__ __forceinline__ void block_reduce_2x8_small(const float (&a)[8], const float (&b)[8], int C, float* __restrict__ s_tot) {
  __shared__ float sh[BN_THREADS * 8];  // [rows][C] with rows*C = 256*8
  const int CG = C >> 3, cg = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float* s0 = sh + (ty * C + cg * 8);
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    if (which) __syncthreads();
    *reinterpret_cast<float4*>(s0) = which ? make_float4(b[0], b[1], b[2], b[3]) : make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(s0 + 4) = which ? make_float4(b[4], b[5], b[6], b[7]) : make_float4(a[4], a[5], a[6], a[7]);
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += BN_THREADS) {
      float acc = 0.f;
      for (int r = 0; r < rows; ++r) acc += sh[r * C + c];
      s_tot[which * C + c] = acc;
    }
  }
}

__device__ __forceinline__ void bn_cluster_emit(const float (&a)[8], const float (&b)[8], int C, BnAcc* __restrict__ acc) {
  extern __shared__ float s_tot[];   // [2*C]
  block_reduce_2x8_small(a, b, C, s_tot);
  cg::cluster_group cluster = cg::this_cluster();
  cluster.sync();
  if (cluster.block_rank() == 0) {
    for (int c = threadIdx.x; c < 2 * C; c += BN_THREADS) {
      float t = s_tot[c];
#pragma unroll
      for (int r = 1; r < BN_CLUSTER; ++r) t += cluster.map_shared_rank(s_tot, r)[c];
      bn_acc_add(acc + c, t);
    }
  }
  cluster.sync();   // the peers' shared memory stays alive until CTA 0 has read it
}

__global__ void __cluster_dims__(BN_CLUSTER, 1, 1) __launch_bounds__(BN_THREADS, BN_RED_MINB)
bn_stats_acc_kernel(const __nv_bfloat16* __restrict__ y, long long P, int C, BnAcc* __restrict__ acc) {
  const int CG = C >> 3, cg_ = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const __nv_bfloat16* yp = y + cg_ * 8;
  const long long step = (long long)gridDim.x * rows;
  const long long us = BN_RED_CONTIG ? rows : step, adv = BN_STATS_U * step;
  for (long long r = (long long)blockIdx.x * (BN_RED_CONTIG ? BN_STATS_U * rows : rows) + ty; r < P; r += adv) {
    if (r + (BN_STATS_U - 1) * us < P) {   // BN_STATS_U independent 16-byte loads in flight per thread
      uint4 v[BN_STATS_U];
#pragma unroll
      for (int u = 0; u < BN_STATS_U; ++u) v[u] = *reinterpret_cast<const uint4*>(yp + (r + u * us) * C);
#pragma unroll
      for (int u = 0; u < BN_STATS_U; ++u) {
        float f[8];
        unpack_bf16x2(v[u].x, f[0], f[1]); unpack_bf16x2(v[u].y, f[2], f[3]); unpack_bf16x2(v[u].z, f[4], f[5]); unpack_bf16x2(v[u].w, f[6], f[7]);
#pragma unroll
        for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] = fmaf(f[j], f[j], q[j]); }
      }
    } else {
      for (int u = 0; u < BN_STATS_U && r + u * us < P; ++u) {
        const Vec8 v = load8(yp + (r + u * us) * C);
#pragma unroll
        for (int j = 0; j < 8; ++j) { s[j] += v.v[j]; q[j] = fmaf(v.v[j], v.v[j], q[j]); }
      }
    }
  }
  bn_cluster_emit(s, q, C, acc);
}

// out = relu?(gamma*xhat + beta [+ residual]) with the batch statistics taken from the accumulators (sum y, sum y^2)
__global__ void __launch_bounds__(BN_THREADS, BN_APPLY_MINB) bn_apply_fwd_acc_kernel(const __nv_bfloat16* __restrict__ y, const BnAcc* __restrict__ acc, long long P,
                                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                     float* __restrict__ running_mean, float* __restrict__ running_var,
                                                                     float momentum, float eps, float* __restrict__ mean_out,
                                                                     float* __restrict__ invstd_out, const __nv_bfloat16* __restrict__ residual,
                                                                     int relu, __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ relu_bits,
                                                                     long long nvec, int C) {
  extern __shared__ float s_coef[];   // [2][C]
  float* s_sc = s_coef;
  float* s_sh = s_coef + C;
  for (int c = threadIdx.x; c < C; c += BN_THREADS) {
    const double n = (double)P;
    const double mean = bn_acc_read(acc + c) / n;
    double var = bn_acc_read(acc + C + c) / n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float g = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
    s_sc[c] = g * invstd;
    s_sh[c] = bt - (float)mean * g * invstd;
    if (blockIdx.x == 0) {
      mean_out[c] = (float)mean;
      invstd_out[c] = invstd;
      if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
      if (running_var) {
        const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
      }
    }
  }
  __syncthreads();
  // the channel group of a thread is the same for every vector it touches: the grid stride is a multiple of 256, 256 of C/8
  const int cg = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) % (C >> 3));
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = s_sc[cg * 8 + j]; sh[j] = s_sh[cg * 8 + j]; }
  auto finish = [&](long long i, const uint4& yu, const uint4& ru) {
    float v[8], o[8];
    unpack_bf16x2(yu.x, v[0], v[1]); unpack_bf16x2(yu.y, v[2], v[3]); unpack_bf16x2(yu.z, v[4], v[5]); unpack_bf16x2(yu.w, v[6], v[7]);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(v[j], sc[j], sh[j]);
    if (residual) {
      float r[8];
      unpack_bf16x2(ru.x, r[0], r[1]); unpack_bf16x2(ru.y, r[2], r[3]); unpack_bf16x2(ru.z, r[4], r[5]); unpack_bf16x2(ru.w, r[6], r[7]);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] += r[j];
    }
    if (relu) {
      if (relu_bits) {
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) m |= (o[j] > 0.f ? 1u : 0u) << j;
        relu_bits[i] = (uint8_t)m;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fmaxf(o[j], 0.f);
    }
    store8(out + i * 8, o);
  };
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long us = BN_APPLY_CONTIG ? BN_THREADS : stride, adv = BN_APPLY_U * stride;
  for (long long i = (long long)blockIdx.x * (BN_APPLY_CONTIG ? BN_APPLY_U * BN_THREADS : BN_THREADS) + threadIdx.x; i < nvec; i += adv) {
    if (i + (BN_APPLY_U - 1) * us < nvec) {   // BN_APPLY_U vectors (x 1-2 loads) in flight per thread
      uint4 yu[BN_APPLY_U], ru[BN_APPLY_U];
#pragma unroll
      for (int u = 0; u < BN_APPLY_U; ++u) {
        yu[u] = *reinterpret_cast<const uint4*>(y + (i + u * us) * 8);
        ru[u] = residual ? *reinterpret_cast<const uint4*>(residual + (i + u * us) * 8) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < BN_APPLY_U; ++u) finish(i + u * us, yu[u], ru[u]);
    } else {
      for (int u = 0; u < BN_APPLY_U && i + u * us < nvec; ++u) {
        const uint4 yu = *reinterpret_cast<const uint4*>(y + (i + u * us) * 8);
        const uint4 ru = residual ? *reinterpret_cast<const uint4*>(residual + (i + u * us) * 8) : make_uint4(0, 0, 0, 0);
        finish(i + u * us, yu, ru);
      }
    }
  }
}

// sum d' and sum d'*xhat per channel (d' = dout masked by the ReLU that followed the BatchNorm).  The loop accumulates the RAW moment
// sum d'*y; xhat = (y - mean)*invstd is applied to the thread's two sums once, after the loop (sum d'*xhat = invstd*(sum d'*y - mean*sum d')
// over the <= 64 rows a thread owns): 16 fewer live registers and two fewer operations per element than normalising every element.
template <bool BITS>
__global__ void __cluster_dims__(BN_CLUSTER, 1, 1) __launch_bounds__(BN_THREADS, BN_RED_MINB)
bn_bwd_acc_kernel(const __nv_bfloat16* __restrict__ dout, const void* __restrict__ out_mask, const __nv_bfloat16* __restrict__ y,
                  const float* __restrict__ mean, const float* __restrict__ invstd, long long P, int C, BnAcc* __restrict__ acc) {
  const int CG = C >> 3, cg_ = threadIdx.x % CG, ty = threadIdx.x / CG, rows = BN_THREADS / CG;
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long step = (long long)gridDim.x * rows;
  const uint8_t* mbits = static_cast<const uint8_t*>(out_mask);
  const __nv_bfloat16* mvals = static_cast<const __nv_bfloat16*>(out_mask);
  auto accumulate = [&](const uint4& du, const uint4& vu, uint32_t m, const uint4& mu4) {
    float d[8], v[8];
    unpack_bf16x2(du.x, d[0], d[1]); unpack_bf16x2(du.y, d[2], d[3]); unpack_bf16x2(du.z, d[4], d[5]); unpack_bf16x2(du.w, d[6], d[7]);
    unpack_bf16x2(vu.x, v[0], v[1]); unpack_bf16x2(vu.y, v[2], v[3]); unpack_bf16x2(vu.z, v[4], v[5]); unpack_bf16x2(vu.w, v[6], v[7]);
    if (out_mask) {
      if constexpr (BITS) {
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = (m >> j) & 1u ? d[j] : 0.f;
      } else {
        float mv[8];
        unpack_bf16x2(mu4.x, mv[0], mv[1]); unpack_bf16x2(mu4.y, mv[2], mv[3]); unpack_bf16x2(mu4.z, mv[4], mv[5]); unpack_bf16x2(mu4.w, mv[6], mv[7]);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = mv[j] > 0.f ? d[j] : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s1[j] += d[j];
      s2[j] = fmaf(d[j], v[j], s2[j]);
    }
  };
  const long long col = cg_ * 8;
  const long long us = BN_RED_CONTIG ? rows : step, adv = BN_BWDRED_U * step;
  for (long long r = (long long)blockIdx.x * (BN_RED_CONTIG ? BN_BWDRED_U * rows : rows) + ty; r < P; r += adv) {
    if (r + (BN_BWDRED_U - 1) * us < P) {   // BN_BWDRED_U rows = 2-3 independent loads each, all issued before the first use
      uint4 du[BN_BWDRED_U], vu[BN_BWDRED_U], mu4[BN_BWDRED_U];
      uint32_t m[BN_BWDRED_U];
#pragma unroll
      for (int u = 0; u < BN_BWDRED_U; ++u) {
        const long long o = (r + u * us) * C + col;
        du[u] = *reinterpret_cast<const uint4*>(dout + o);
        vu[u] = *reinterpret_cast<const uint4*>(y + o);
        m[u] = 0;
        mu4[u] = make_uint4(0, 0, 0, 0);
        if (out_mask) {
          if constexpr (BITS) m[u] = mbits[o >> 3];
          else mu4[u] = *reinterpret_cast<const uint4*>(mvals + o);
        }
      }
#pragma unroll
      for (int u = 0; u < BN_BWDRED_U; ++u) accumulate(du[u], vu[u], m[u], mu4[u]);
    } else {
      for (int u = 0; u < BN_BWDRED_U && r + u * us < P; ++u) {
        const long long o = (r + u * us) * C + col;
        const uint4 du = *reinterpret_cast<const uint4*>(dout + o);
        const uint4 vu = *reinterpret_cast<const uint4*>(y + o);
        uint32_t m = 0;
        uint4 mu4 = make_uint4(0, 0, 0, 0);
        if (out_mask) {
          if constexpr (BITS) m = mbits[o >> 3];
          else mu4 = *reinterpret_cast<const uint4*>(mvals + o);
        }
        accumulate(du, vu, m, mu4);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) s2[j] = invstd[col + j] * fmaf(-mean[col + j], s1[j], s2[j]);
  bn_cluster_emit(s1, s2, C, acc);
}

template <bool BITS>
__global__ void __launch_bounds__(BN_THREADS, BN_APPLY_MINB) bn_bwd_apply_acc_kernel(const __nv_bfloat16* __restrict__ dout, const void* __restrict__ out_mask,
                                                                     const __nv_bfloat16* __restrict__ y, const float* __restrict__ mean,
                                                                     const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                                     const BnAcc* __restrict__ acc, long long P, float* __restrict__ dgamma,
                                                                     float* __restrict__ dbeta, int accumulate, __nv_bfloat16* __restrict__ dy,
                                                                     __nv_bfloat16* __restrict__ dmasked, long long nvec, int C) {
  extern __shared__ float s_k3[];   // [3][C]
  float* s_k[3] = {s_k3, s_k3 + C, s_k3 + 2 * C};
  for (int c = threadIdx.x; c < C; c += BN_THREADS) {
    const double s1 = bn_acc_read(acc + c), s2 = bn_acc_read(acc + C + c);
    const float a = (gamma ? gamma[c] : 1.f) * invstd[c];
    const float c1 = (float)(s1 / (double)P), c2 = (float)(s2 / (double)P);
    const float k1 = -a * c2 * invstd[c];
    s_k[0][c] = a;
    s_k[1][c] = k1;
    s_k[2][c] = -a * c1 - k1 * mean[c];
    if (blockIdx.x == 0) {
      if (dbeta) dbeta[c] = (accumulate ? dbeta[c] : 0.f) + (float)s1;
      if (dgamma) dgamma[c] = (accumulate ? dgamma[c] : 0.f) + (float)s2;
    }
  }
  __syncthreads();
  // The channel group of a thread is the same for every vector it touches (the grid stride is a multiple of 256, 256 of C/8).  Its 24
  // coefficients stay in shared memory and are re-read (six 16-byte loads) once per batch of BN_APPLY_U vectors: held in registers they
  // cost 24 of the registers that decide how many blocks are resident, and this kernel's throughput is the bytes it keeps in flight.
  const int c0 = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) % (C >> 3)) * 8;
  const float4* kk0 = reinterpret_cast<const float4*>(s_k[0] + c0);
  const float4* kk1 = reinterpret_cast<const float4*>(s_k[1] + c0);
  const float4* kk2 = reinterpret_cast<const float4*>(s_k[2] + c0);
  const uint8_t* mbits = static_cast<const uint8_t*>(out_mask);
  const __nv_bfloat16* mvals = static_cast<const __nv_bfloat16*>(out_mask);
  auto finish = [&](long long i, const uint4& du, const uint4& vu, uint32_t m, const uint4& mu4) {
    float d[8], v[8];
    unpack_bf16x2(du.x, d[0], d[1]); unpack_bf16x2(du.y, d[2], d[3]); unpack_bf16x2(du.z, d[4], d[5]); unpack_bf16x2(du.w, d[6], d[7]);
    unpack_bf16x2(vu.x, v[0], v[1]); unpack_bf16x2(vu.y, v[2], v[3]); unpack_bf16x2(vu.z, v[4], v[5]); unpack_bf16x2(vu.w, v[6], v[7]);
    if (out_mask) {
      if constexpr (BITS) {
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = (m >> j) & 1u ? d[j] : 0.f;
      } else {
        float mv[8];
        unpack_bf16x2(mu4.x, mv[0], mv[1]); unpack_bf16x2(mu4.y, mv[2], mv[3]); unpack_bf16x2(mu4.z, mv[4], mv[5]); unpack_bf16x2(mu4.w, mv[6], mv[7]);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = mv[j] > 0.f ? d[j] : 0.f;
      }
    }
    if (dmasked) store8(dmasked + i * 8, d);
    const float4 a0 = kk0[0], a1 = kk0[1], b0 = kk1[0], b1 = kk1[1], g0 = kk2[0], g1 = kk2[1];
    const float k0[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float k1[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    const float k2[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(k0[j], d[j], fmaf(k1[j], v[j], k2[j]));
    store8(dy + i * 8, o);
  };
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long us = BN_APPLY_CONTIG ? BN_THREADS : stride, adv = BN_APPLY_U * stride;
  for (long long i = (long long)blockIdx.x * (BN_APPLY_CONTIG ? BN_APPLY_U * BN_THREADS : BN_THREADS) + threadIdx.x; i < nvec; i += adv) {
    if (i + (BN_APPLY_U - 1) * us < nvec) {
      uint4 du[BN_APPLY_U], vu[BN_APPLY_U], mu4[BN_APPLY_U];
      uint32_t m[BN_APPLY_U];
#pragma unroll
      for (int u = 0; u < BN_APPLY_U; ++u) {
        const long long iu = i + u * us;
        du[u] = *reinterpret_cast<const uint4*>(dout + iu * 8);
        vu[u] = *reinterpret_cast<const uint4*>(y + iu * 8);
        m[u] = 0;
        mu4[u] = make_uint4(0, 0, 0, 0);
        if (out_mask) {
          if constexpr (BITS) m[u] = mbits[iu];
          else mu4[u] = *reinterpret_cast<const uint4*>(mvals + iu * 8);
        }
      }
#pragma unroll
      for (int u = 0; u < BN_APPLY_U; ++u) finish(i + u * us, du[u], vu[u], m[u], mu4[u]);
    } else {
      for (int u = 0; u < BN_APPLY_U && i + u * us < nvec; ++u) {
        const long long iu = i + u * us;
        const uint4 du = *reinterpret_cast<const uint4*>(dout + iu * 8);
        const uint4 vu = *reinterpret_cast<const uint4*>(y + iu * 8);
        uint32_t m = 0;
        uint4 mu4 = make_uint4(0, 0, 0, 0);
        if (out_mask) {
          if constexpr (BITS) m = mbits[iu];
          else mu4 = *reinterpret_cast<const uint4*>(mvals + iu * 8);
        }
        finish(iu, du, vu, m, mu4);
      }
    }
  }
}

static int bn_grid_rows(long long P, int C) {
  const int rows = BN_THREADS / (C >> 3);
  long long blocks = ceil_div_ll(P, (long long)rows * 16);  // >= 16 row iterations per block: few partials to finalize
  if (blocks > BN_MAX_BLOCKS) blocks = BN_MAX_BLOCKS;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}
static int bn_grid_elems(long long nvec) {
  long long blocks = ceil_div_ll(nvec, BN_THREADS);
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  return (int)blocks;
}
// Grid of the reduce kernels: a whole number of 8-CTA clusters, at most ONE resident wave.  "Resident" is asked of
// cudaOccupancyMaxActiveClusters, not derived from blocks per SM x SMs: a cluster lives inside one GPC, so a grid that fills every
// block slot of the GPU only fits if every GPC's slot count is a multiple of 8 -- otherwise the last clusters wait for a second wave and
// the kernel takes up to twice as long (measured: the 592-block grid at exactly 4 blocks per SM ran 25 % slower than the same grid with
// a fifth slot free).  One wave less one cluster per GPC's worth of slack keeps every cluster co-resident.
template <int TAG, class K>   // TAG: one cached answer per kernel instantiation and channel count (instantiations may share a function type)
static int bn_grid_acc_rows(K kernel, long long P, int C, size_t smem, int U) {
  static int resident_by_c[12] = {0};   // index: log2(C)
  int lg = 0;
  while ((1 << lg) < C && lg < 11) ++lg;
  int& resident = resident_by_c[lg];
  if (resident == 0) {
    int clusters = 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(BN_CLUSTER * (unsigned)sm_count(), 1, 1);
    cfg.blockDim = dim3(BN_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = BN_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg) == cudaSuccess && clusters > 0) {
      resident = clusters * BN_CLUSTER;
    } else {
      (void)cudaGetLastError();
      int occ = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, BN_THREADS, smem) != cudaSuccess || occ < 1) occ = 2;
      resident = (occ * sm_count() / BN_CLUSTER - 8) * BN_CLUSTER;   // one cluster of slack per GPC
    }
    if (resident > BN_ACC_MAX_BLOCKS) resident = BN_ACC_MAX_BLOCKS;
    if (resident < BN_CLUSTER) resident = BN_CLUSTER;
  }
  // equal shares: chunks of U x rows rows (U = the rows a thread has in flight), at least four per block, the same number (+-1) for every block
  const int rows = BN_THREADS / (C >> 3);
  const long long chunks = ceil_div_ll(P, (long long)rows * U);
  long long gmax = ceil_div_ll(chunks, BN_RED_MIN_CHUNKS);
  if (gmax > resident) gmax = resident;
  const long long iters = ceil_div_ll(chunks, gmax);
  long long blocks = ceil_div_ll(ceil_div_ll(chunks, iters), BN_CLUSTER) * BN_CLUSTER;
  if (blocks > resident) blocks = resident;
  return (int)blocks;
}
// Grid of the accumulator apply kernels.  Every block pays the coefficient prologue, so few fat blocks.  The work is split into chunks of
// BN_APPLY_U x 256 vectors; the grid is the smallest one that gives every block the same number of chunks (+-1) within BN_APPLY_WAVES
// resident waves -- a grid-stride loop over unequal shares waits for its slowest block (a 1184-block grid at 5 resident blocks per SM ran
// a full wave plus a 3/5 one: 1.4x the time of the 16-blocks-per-SM grid it replaced).
#ifndef BN_APPLY_WAVES
#define BN_APPLY_WAVES 1
#endif
template <int TAG, class K>
static int bn_grid_apply(K kernel, long long nvec, size_t smem) {
  static int resident = 0;   // per kernel instantiation
  if (resident == 0) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, BN_THREADS, smem) != cudaSuccess || occ < 1) occ = 4;
    resident = occ * sm_count();
  }
  const long long chunks = ceil_div_ll(nvec, (long long)BN_THREADS * BN_APPLY_U);
  const long long gmax = (long long)BN_APPLY_WAVES * resident;
  const long long iters = ceil_div_ll(chunks, gmax);
  long long blocks = ceil_div_ll(chunks, iters);
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}
static bool bn_c_ok(int C) { return C >= 8 && C <= 2048 && (C & 7) == 0 && (BN_THREADS % (C >> 3)) == 0; }

// ================================================================================================================================
// Frozen BatchNorm: a BatchNorm module in eval() mode inside a train()-mode model (fine-tuning with frozen BN, as torchvision's
// detection and keypoint models do).  torch then normalises with the running statistics, which are constants of the step:
//   forward : out = relu?(scale*y + shift [+ residual]),  scale = gamma*invstd_r, shift = beta - mean_r*scale (bn_fold_kernel)
//   backward: d' = dout*[out>0];  dy = scale*d'  -- no batch-statistics terms;  dbeta = sum d',  dgamma = sum d'*(y - mean_r)*invstd_r
// The backward is one pass.  Where gamma or beta is trained it adds (sum d', sum d'*y) into the 128-bit accumulators of hk_bn_acc.cuh
// and the last cluster to retire derives dgamma = invstd_r*(sum d'*y - mean_r*sum d') and dbeta = sum d' from the exact totals
// (deterministic, no finalize launch).  The retire counter is the spare word of the first accumulator (zero with the accumulators).

// per-channel fold of every frozen BatchNorm of a step in one launch: blockIdx.y = item
__global__ void __launch_bounds__(256) bn_fold_kernel(const HkBnFoldItem* __restrict__ items) {
  const HkBnFoldItem it = items[blockIdx.y];
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= it.C) return;
  const float invstd = (float)(1.0 / sqrt((double)it.var[c] + (double)it.eps));
  const float g = it.gamma ? it.gamma[c] : 1.f, bt = it.beta ? it.beta[c] : 0.f;
  const float sc = g * invstd;
  it.scale[c] = sc;
  it.shift[c] = bt - it.mean[c] * sc;
  if (it.invstd) it.invstd[c] = invstd;
}

// accumulator totals written by other CTAs' atomics: read through L2
__device__ __forceinline__ double bn_acc_read_l2(const BnAcc* a) {
  BnAcc v;
  v.lo = __ldcg(&a->lo);
  v.hi = __ldcg(&a->hi);
  v.poison = __ldcg(&a->poison);
  return bn_acc_read(&v);
}

// The bf16-mask variant keeps a third 16-byte operand per vector in flight: held to BN_APPLY_MINB blocks per SM it spills, so it runs
// at one resident block fewer.
template <bool BITS>
__global__ void __cluster_dims__(BN_CLUSTER, 1, 1) __launch_bounds__(BN_THREADS, BITS ? BN_APPLY_MINB : BN_APPLY_MINB - 1)
bn_frozen_bwd_kernel(const __nv_bfloat16* __restrict__ dout, const void* __restrict__ out_mask, const __nv_bfloat16* __restrict__ y,
                     const float* __restrict__ scale, const float* __restrict__ mean, const float* __restrict__ invstd,
                     BnAcc* __restrict__ acc, float* __restrict__ dgamma, float* __restrict__ dbeta, int accumulate,
                     __nv_bfloat16* __restrict__ dy, __nv_bfloat16* __restrict__ dmasked, long long nvec, int C) {
  // the channel group of a thread is the same for every vector it touches (the grid stride is a multiple of 256, 256 of C/8), and it is
  // the one block_reduce_2x8_small expects (threadIdx % (C/8))
  const int c0 = (threadIdx.x % (C >> 3)) * 8;
  float k[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) k[j] = __ldg(scale + c0 + j);
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const bool sums = acc != nullptr;
  const uint8_t* mbits = static_cast<const uint8_t*>(out_mask);
  const __nv_bfloat16* mvals = static_cast<const __nv_bfloat16*>(out_mask);
  auto finish = [&](long long i, const uint4& du, uint32_t m, const uint4& mu4, const uint4& vu) {
    float d[8];
    unpack_bf16x2(du.x, d[0], d[1]); unpack_bf16x2(du.y, d[2], d[3]); unpack_bf16x2(du.z, d[4], d[5]); unpack_bf16x2(du.w, d[6], d[7]);
    if (out_mask) {
      if constexpr (BITS) {
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = (m >> j) & 1u ? d[j] : 0.f;
      } else {
        float mv[8];
        unpack_bf16x2(mu4.x, mv[0], mv[1]); unpack_bf16x2(mu4.y, mv[2], mv[3]); unpack_bf16x2(mu4.z, mv[4], mv[5]); unpack_bf16x2(mu4.w, mv[6], mv[7]);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = mv[j] > 0.f ? d[j] : 0.f;
      }
    }
    if (dmasked) store8(dmasked + i * 8, d);
    if (dy) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = k[j] * d[j];
      store8(dy + i * 8, o);
    }
    if (sums) {
      float v[8];
      unpack_bf16x2(vu.x, v[0], v[1]); unpack_bf16x2(vu.y, v[2], v[3]); unpack_bf16x2(vu.z, v[4], v[5]); unpack_bf16x2(vu.w, v[6], v[7]);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s1[j] += d[j]; s2[j] = fmaf(d[j], v[j], s2[j]); }
    }
  };
  auto load = [&](long long iu, uint4& du, uint32_t& m, uint4& mu4, uint4& vu) {
    du = *reinterpret_cast<const uint4*>(dout + iu * 8);
    vu = sums ? *reinterpret_cast<const uint4*>(y + iu * 8) : make_uint4(0, 0, 0, 0);
    m = 0;
    mu4 = make_uint4(0, 0, 0, 0);
    if (out_mask) {
      if constexpr (BITS) m = mbits[iu];
      else mu4 = *reinterpret_cast<const uint4*>(mvals + iu * 8);
    }
  };
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long us = BN_APPLY_CONTIG ? BN_THREADS : stride, adv = BN_APPLY_U * stride;
  for (long long i = (long long)blockIdx.x * (BN_APPLY_CONTIG ? BN_APPLY_U * BN_THREADS : BN_THREADS) + threadIdx.x; i < nvec; i += adv) {
    if (i + (BN_APPLY_U - 1) * us < nvec) {   // BN_APPLY_U vectors (x 1-3 loads) in flight per thread
      uint4 du[BN_APPLY_U], mu4[BN_APPLY_U], vu[BN_APPLY_U];
      uint32_t m[BN_APPLY_U];
#pragma unroll
      for (int u = 0; u < BN_APPLY_U; ++u) load(i + u * us, du[u], m[u], mu4[u], vu[u]);
#pragma unroll
      for (int u = 0; u < BN_APPLY_U; ++u) finish(i + u * us, du[u], m[u], mu4[u], vu[u]);
    } else {
      for (int u = 0; u < BN_APPLY_U && i + u * us < nvec; ++u) {
        uint4 du, mu4, vu;
        uint32_t m;
        load(i + u * us, du, m, mu4, vu);
        finish(i + u * us, du, m, mu4, vu);
      }
    }
  }
  if (!sums) return;
  bn_cluster_emit(s1, s2, C, acc);
  if (cg::this_cluster().block_rank() != 0) return;
  // CTA 0 of every cluster has issued its cluster's atomics: the last one to get here turns the totals into dgamma / dbeta.  The flag
  // lives in the dynamic buffer of bn_cluster_emit, free after its final cluster barrier (a static __shared__ variable here could be
  // placed ahead of block_reduce_2x8_small's buffer and break the alignment of its float4 stores).
  extern __shared__ float s_tot[];
  volatile int* last = reinterpret_cast<volatile int*>(s_tot);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) *last = atomicAdd(&acc[0].pad, 1ull) == (unsigned long long)(gridDim.x / BN_CLUSTER - 1) ? 1 : 0;
  __syncthreads();
  if (!*last) return;
  __threadfence();
  for (int c = threadIdx.x; c < C; c += BN_THREADS) {
    const double t1 = bn_acc_read_l2(acc + c), t2 = bn_acc_read_l2(acc + C + c);
    if (dbeta) dbeta[c] = (accumulate ? dbeta[c] : 0.f) + (float)t1;
    if (dgamma) dgamma[c] = (accumulate ? dgamma[c] : 0.f) + (float)((double)invstd[c] * (t2 - (double)mean[c] * t1));
  }
  if (threadIdx.x == 0) acc[0].pad = 0;   // the buffer can be cleared and reused as before
}

// Grid of the frozen backward: chunks of BN_APPLY_U x 256 vectors shared equally (as bn_grid_apply), in whole 8-CTA clusters, at most one
// resident wave of clusters (cudaOccupancyMaxActiveClusters, see bn_grid_acc_rows).
template <int TAG, class K>
static int bn_grid_frozen(K kernel, long long nvec, size_t smem) {
  static int resident_by_dev[64] = {0};
  int dev = 0;
  (void)cudaGetDevice(&dev);
  int fallback = 0;
  int& resident = dev < 64 ? resident_by_dev[dev] : fallback;
  if (resident == 0) {
    int clusters = 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(BN_CLUSTER * (unsigned)sm_count(), 1, 1);
    cfg.blockDim = dim3(BN_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = BN_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg) == cudaSuccess && clusters > 0) {
      resident = clusters * BN_CLUSTER;
    } else {
      (void)cudaGetLastError();
      int occ = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, BN_THREADS, smem) != cudaSuccess || occ < 1) occ = 2;
      resident = (occ * sm_count() / BN_CLUSTER - 8) * BN_CLUSTER;
    }
    if (resident < BN_CLUSTER) resident = BN_CLUSTER;
  }
  const long long chunks = ceil_div_ll(nvec, (long long)BN_THREADS * BN_APPLY_U);
  const long long iters = ceil_div_ll(chunks, resident);
  long long blocks = ceil_div_ll(ceil_div_ll(chunks, iters), BN_CLUSTER) * BN_CLUSTER;
  if (blocks > resident) blocks = resident;
  if (blocks < BN_CLUSTER) blocks = BN_CLUSTER;
  return (int)blocks;
}

}  // namespace hk

extern "C" {

size_t hk_bn_workspace_bytes(int C) { return (size_t)hk::BN_MAX_BLOCKS * 2 * (size_t)C * sizeof(float); }

int hk_bn_train_stats(const void* y, long long P, int C, const float* gamma, const float* beta, float* running_mean,
                      float* running_var, float momentum, float eps, float* mean_out, float* invstd_out, float* scale_out,
                      float* shift_out, void* ws, size_t ws_bytes, void* stream) {
  using namespace hk;
  HK_REQUIRE(y && mean_out && invstd_out && scale_out && shift_out && ws, "hk_bn_train_stats: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_train_stats: unsupported shape P=%lld C=%d (C must be a power-of-two multiple of 8 up to 2048)", P, C);
  HK_REQUIRE(ws_bytes >= hk_bn_workspace_bytes(C), "hk_bn_train_stats: workspace too small");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(y) & 15) == 0, "hk_bn_train_stats: y must be 16-byte aligned");
  const int blocks = bn_grid_rows(P, C);
  bn_stats_partial_kernel<<<blocks, BN_THREADS, 0, as_stream(stream)>>>(static_cast<const __nv_bfloat16*>(y), P, C, static_cast<float*>(ws));
  int rc = check_launch("bn_stats_partial_kernel");
  if (rc) return rc;
  bn_stats_finalize_kernel<<<ceil_div(C, 32), BN_FIN_THREADS, 0, as_stream(stream)>>>(static_cast<const float*>(ws), blocks, P, C, gamma, beta,
                                                                           running_mean, running_var, momentum, eps, mean_out,
                                                                           invstd_out, scale_out, shift_out);
  return check_launch("bn_stats_finalize_kernel");
}

int hk_bn_apply_fwd(const void* y, const float* scale, const float* shift, const void* residual_or_null, int relu, void* out,
                    void* relu_bits_or_null, long long P, int C, void* stream) {
  using namespace hk;
  HK_REQUIRE(y && scale && shift && out, "hk_bn_apply_fwd: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_apply_fwd: unsupported shape P=%lld C=%d (C must be a power-of-two multiple of 8 up to 2048)", P, C);
  const long long nvec = P * (C >> 3);
  bn_apply_fwd_kernel<<<bn_grid_elems(nvec), BN_THREADS, 0, as_stream(stream)>>>(
      static_cast<const __nv_bfloat16*>(y), scale, shift, static_cast<const __nv_bfloat16*>(residual_or_null), relu,
      static_cast<__nv_bfloat16*>(out), static_cast<uint8_t*>(relu_bits_or_null), nvec, C);
  return check_launch("bn_apply_fwd_kernel");
}

int hk_bn_train_bwd(const void* dout, const void* out_mask_or_null, int mask_is_bits, const void* y, const float* mean, const float* invstd,
                    const float* gamma, long long P, int C, float* dgamma, float* dbeta, int accumulate, void* dy,
                    void* dmasked_or_null, void* ws, size_t ws_bytes, void* stream) {
  using namespace hk;
  HK_REQUIRE(dout && y && mean && invstd && dy && ws, "hk_bn_train_bwd: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_train_bwd: unsupported shape P=%lld C=%d", P, C);
  HK_REQUIRE(ws_bytes >= hk_bn_workspace_bytes(C) + 3 * (size_t)C * sizeof(float), "hk_bn_train_bwd: workspace too small");
  const int blocks = bn_grid_rows(P, C);
  float* partial = static_cast<float*>(ws);
  float* coef = partial + (size_t)BN_MAX_BLOCKS * 2 * C;
  const __nv_bfloat16* d = static_cast<const __nv_bfloat16*>(dout);
  const void* m = out_mask_or_null;
  const __nv_bfloat16* yy = static_cast<const __nv_bfloat16*>(y);
  if (mask_is_bits) bn_bwd_partial_kernel<true><<<blocks, BN_THREADS, 0, as_stream(stream)>>>(d, m, yy, mean, invstd, P, C, partial);
  else bn_bwd_partial_kernel<false><<<blocks, BN_THREADS, 0, as_stream(stream)>>>(d, m, yy, mean, invstd, P, C, partial);
  int rc = check_launch("bn_bwd_partial_kernel");
  if (rc) return rc;
  bn_bwd_finalize_kernel<<<ceil_div(C, 32), BN_FIN_THREADS, 0, as_stream(stream)>>>(partial, blocks, P, C, gamma, invstd, dgamma, dbeta, accumulate, coef);
  rc = check_launch("bn_bwd_finalize_kernel");
  if (rc) return rc;
  const long long nvec = P * (C >> 3);
  if (mask_is_bits)
    bn_bwd_apply_kernel<true><<<bn_grid_elems(nvec), BN_THREADS, 0, as_stream(stream)>>>(d, m, yy, mean, invstd, coef, static_cast<__nv_bfloat16*>(dy),
                                                                                       static_cast<__nv_bfloat16*>(dmasked_or_null), nvec, C);
  else
    bn_bwd_apply_kernel<false><<<bn_grid_elems(nvec), BN_THREADS, 0, as_stream(stream)>>>(d, m, yy, mean, invstd, coef, static_cast<__nv_bfloat16*>(dy),
                                                                                        static_cast<__nv_bfloat16*>(dmasked_or_null), nvec, C);
  return check_launch("bn_bwd_apply_kernel");
}

size_t hk_bn_acc_bytes(int C) { return 2 * (size_t)C * sizeof(hk::BnAcc); }

int hk_bn_stats_acc(const void* y, long long P, int C, void* acc, void* stream) {
  using namespace hk;
  HK_REQUIRE(y && acc, "hk_bn_stats_acc: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_stats_acc: unsupported shape P=%lld C=%d (C must be a power-of-two multiple of 8 up to 2048)", P, C);
  HK_REQUIRE((reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(acc) & 31) == 0, "hk_bn_stats_acc: misaligned buffer");
  bn_stats_acc_kernel<<<bn_grid_acc_rows<0>(bn_stats_acc_kernel, P, C, 2 * (size_t)C * 4, BN_STATS_U), BN_THREADS, 2 * (size_t)C * 4, as_stream(stream)>>>(static_cast<const __nv_bfloat16*>(y), P, C, static_cast<BnAcc*>(acc));
  return check_launch("bn_stats_acc_kernel");
}

int hk_bn_apply_fwd_acc(const void* y, const void* acc, long long P, int C, const float* gamma, const float* beta, float* running_mean,
                        float* running_var, float momentum, float eps, float* mean_out, float* invstd_out, const void* residual_or_null,
                        int relu, void* out, void* relu_bits_or_null, void* stream) {
  using namespace hk;
  HK_REQUIRE(y && acc && mean_out && invstd_out && out, "hk_bn_apply_fwd_acc: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_apply_fwd_acc: unsupported shape P=%lld C=%d", P, C);
  const long long nvec = P * (C >> 3);
  bn_apply_fwd_acc_kernel<<<bn_grid_apply<0>(bn_apply_fwd_acc_kernel, nvec, 2 * (size_t)C * 4), BN_THREADS, 2 * (size_t)C * 4, as_stream(stream)>>>(
      static_cast<const __nv_bfloat16*>(y), static_cast<const BnAcc*>(acc), P, gamma, beta, running_mean, running_var, momentum, eps, mean_out,
      invstd_out, static_cast<const __nv_bfloat16*>(residual_or_null), relu, static_cast<__nv_bfloat16*>(out),
      static_cast<uint8_t*>(relu_bits_or_null), nvec, C);
  return check_launch("bn_apply_fwd_acc_kernel");
}

int hk_bn_bwd_acc(const void* dout, const void* out_mask_or_null, int mask_is_bits, const void* y, const float* mean, const float* invstd,
                  const float* gamma, long long P, int C, void* acc, float* dgamma, float* dbeta, int accumulate, void* dy,
                  void* dmasked_or_null, void* stream) {
  using namespace hk;
  HK_REQUIRE(dout && y && mean && invstd && dy && acc, "hk_bn_bwd_acc: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_bwd_acc: unsupported shape P=%lld C=%d", P, C);
  HK_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 31) == 0, "hk_bn_bwd_acc: misaligned accumulator buffer");
  const __nv_bfloat16* d = static_cast<const __nv_bfloat16*>(dout);
  const __nv_bfloat16* yy = static_cast<const __nv_bfloat16*>(y);
  BnAcc* a = static_cast<BnAcc*>(acc);
  const int blocks = mask_is_bits ? bn_grid_acc_rows<1>(bn_bwd_acc_kernel<true>, P, C, 2 * (size_t)C * 4, BN_BWDRED_U) : bn_grid_acc_rows<2>(bn_bwd_acc_kernel<false>, P, C, 2 * (size_t)C * 4, BN_BWDRED_U);
  if (mask_is_bits) bn_bwd_acc_kernel<true><<<blocks, BN_THREADS, 2 * (size_t)C * 4, as_stream(stream)>>>(d, out_mask_or_null, yy, mean, invstd, P, C, a);
  else bn_bwd_acc_kernel<false><<<blocks, BN_THREADS, 2 * (size_t)C * 4, as_stream(stream)>>>(d, out_mask_or_null, yy, mean, invstd, P, C, a);
  int rc = check_launch("bn_bwd_acc_kernel");
  if (rc) return rc;
  const long long nvec = P * (C >> 3);
  const int ablocks = mask_is_bits ? bn_grid_apply<1>(bn_bwd_apply_acc_kernel<true>, nvec, 3 * (size_t)C * 4) : bn_grid_apply<2>(bn_bwd_apply_acc_kernel<false>, nvec, 3 * (size_t)C * 4);
  if (mask_is_bits)
    bn_bwd_apply_acc_kernel<true><<<ablocks, BN_THREADS, 3 * (size_t)C * 4, as_stream(stream)>>>(d, out_mask_or_null, yy, mean, invstd, gamma, a, P, dgamma, dbeta, accumulate,
                                                                               static_cast<__nv_bfloat16*>(dy), static_cast<__nv_bfloat16*>(dmasked_or_null), nvec, C);
  else
    bn_bwd_apply_acc_kernel<false><<<ablocks, BN_THREADS, 3 * (size_t)C * 4, as_stream(stream)>>>(d, out_mask_or_null, yy, mean, invstd, gamma, a, P, dgamma, dbeta, accumulate,
                                                                                static_cast<__nv_bfloat16*>(dy), static_cast<__nv_bfloat16*>(dmasked_or_null), nvec, C);
  return check_launch("bn_bwd_apply_acc_kernel");
}

int hk_bn_fold(const HkBnFoldItem* items_dev, int n_items, int max_c, void* stream) {
  using namespace hk;
  HK_REQUIRE(items_dev && n_items > 0 && n_items <= 65535 && max_c > 0, "hk_bn_fold: bad argument");
  bn_fold_kernel<<<dim3(ceil_div(max_c, 256), n_items), 256, 0, as_stream(stream)>>>(items_dev);
  return check_launch("bn_fold_kernel");
}

int hk_bn_frozen_bwd(const void* dout, const void* out_mask_or_null, int mask_is_bits, const void* y_or_null, const float* scale,
                     const float* mean, const float* invstd, long long P, int C, void* acc_or_null, float* dgamma, float* dbeta,
                     int accumulate, void* dy_or_null, void* dmasked_or_null, void* stream) {
  using namespace hk;
  HK_REQUIRE(dout && scale, "hk_bn_frozen_bwd: null pointer");
  HK_REQUIRE(P > 0 && bn_c_ok(C), "hk_bn_frozen_bwd: unsupported shape P=%lld C=%d", P, C);
  const bool sums = dgamma || dbeta;
  HK_REQUIRE(!sums || (acc_or_null && y_or_null && mean && invstd), "hk_bn_frozen_bwd: dgamma/dbeta need y, mean, invstd and an accumulator buffer");
  HK_REQUIRE(!acc_or_null || (reinterpret_cast<uintptr_t>(acc_or_null) & 31) == 0, "hk_bn_frozen_bwd: misaligned accumulator buffer");
  HK_REQUIRE(sums || dy_or_null || dmasked_or_null, "hk_bn_frozen_bwd: nothing to compute");
  const long long nvec = P * (C >> 3);
  BnAcc* a = sums ? static_cast<BnAcc*>(acc_or_null) : nullptr;
  const size_t smem = 2 * (size_t)C * 4;
  const __nv_bfloat16* d = static_cast<const __nv_bfloat16*>(dout);
  const __nv_bfloat16* yy = static_cast<const __nv_bfloat16*>(y_or_null);
  __nv_bfloat16* dyp = static_cast<__nv_bfloat16*>(dy_or_null);
  __nv_bfloat16* dm = static_cast<__nv_bfloat16*>(dmasked_or_null);
  if (mask_is_bits)
    bn_frozen_bwd_kernel<true><<<bn_grid_frozen<1>(bn_frozen_bwd_kernel<true>, nvec, smem), BN_THREADS, smem, as_stream(stream)>>>(
        d, out_mask_or_null, yy, scale, mean, invstd, a, dgamma, dbeta, accumulate, dyp, dm, nvec, C);
  else
    bn_frozen_bwd_kernel<false><<<bn_grid_frozen<2>(bn_frozen_bwd_kernel<false>, nvec, smem), BN_THREADS, smem, as_stream(stream)>>>(
        d, out_mask_or_null, yy, scale, mean, invstd, a, dgamma, dbeta, accumulate, dyp, dm, nvec, C);
  return check_launch("bn_frozen_bwd_kernel");
}

}  // extern "C"
