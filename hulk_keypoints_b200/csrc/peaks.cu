// Every keypoint instance of a heatmap channel: thresholded local maxima, the top N per (H, W) map.
//
// Pixel p with value v is a peak iff v >= threshold, v > q for every neighbour q of its (2r+1)x(2r+1) window (clipped to the image)
// that comes before p in row-major order, and v >= q for every neighbour after p.  NaN reads as -inf, so with a finite threshold NaN and
// -inf pixels are never peaks and never suppress one.  On a plateau only the first pixel survives; the top-1 peak is the first maximum,
// i.e. what hk_argmax_decode returns on a NaN-free map.
//
// Separable form of the same test (O(r) compares per pixel instead of O(r^2)):
//   Mrow(y,x) = max v over columns [x-r, x+r] of row y      L  = max v over columns [x-r, x-1] of row y
//   U         = max Mrow over rows [y-r, y-1]               Dn = max Mrow over rows [y, y+r]
//   peak  <=>  v >= threshold && v >= max(U, Dn) && v > max(U, L)
//
// Two launches, no global atomics, output independent of scheduling:
//   1. peak_tile_kernel<r>, grid (tiles, B*K): one 32x128 output tile plus its r-pixel halo in shared memory (one HBM read of the map;
//      the halo re-reads hit L2).  Rows pass: Mrow for every halo row and the row half of the test (v >= thr, v >= Mrow, v > L) for
//      the tile's pixels; columns pass: U and Dn for the pixels that survived.  Each peak becomes the 64-bit key
//      (orderable(v) << 32) | ~flat_index -- larger key = higher value, then lower index; keys are unique -- appended to a shared list
//      in any order; a bitonic sort makes the list's order (and so the output) independent of that.  The top min(N, count) keys go to
//      the workspace with their count.
//   2. peak_merge_kernel, one CTA per map: merges the tiles' sorted lists into the map's top N (the global top N is contained in the
//      union of the per-tile top-N lists), reading only the filled slots, and writes yx / score / count and the padding.
#include "hk_common.cuh"

namespace hk {

constexpr int kPeakTH = 32, kPeakTW = 128, kPeakThreads = 256;
constexpr int kPeakMaxN = 256, kPeakMaxR = 16;
// two peaks are more than r >= 1 apart in both axes (each is in the other's window, and the strict / non-strict rule cannot hold both
// ways), so a 2x2 block holds at most one: a tile has at most 16 x 64 peaks
constexpr int kPeakMaxTileKeys = (kPeakTH / 2) * (kPeakTW / 2);
constexpr int kPeakRowRun = 8;                                          // columns per thread in the rows pass
constexpr int kPeakColRun = kPeakTH * kPeakTW / kPeakThreads;           // rows per thread in the columns pass (16)
static_assert(kPeakTH % kPeakColRun == 0 && kPeakTW % kPeakRowRun == 0, "tile shape");

typedef unsigned long long u64;

// monotone map float -> uint32 (-0 and +0 map alike, so equal values tie on the flat index as the definition asks)
__device__ __forceinline__ uint32_t peak_orderable(float v) {
  const uint32_t u = v == 0.0f ? 0u : __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float peak_value(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }

__device__ __forceinline__ float nan_to_ninf(float v) { return v != v ? -INFINITY : v; }

template <int R>
struct PeakTile {
  static constexpr int R4 = (R + 3) & ~3;                 // halo columns, rounded up so raw rows stay float4-aligned
  static constexpr int rows = kPeakTH + 2 * R;            // halo rows
  static constexpr int pitch = kPeakTW + 2 * R4;          // floats per raw row
  static constexpr int keys_off = 0;
  static constexpr int raw_off = kPeakMaxTileKeys * 8;
  static constexpr int mrow_off = raw_off + rows * pitch * 4;
  static constexpr int flag_off = mrow_off + rows * kPeakTW * 4;
  static constexpr int bytes = flag_off + kPeakTH * kPeakTW;
};

template <int R>
__global__ void __launch_bounds__(kPeakThreads)
peak_tile_kernel(const float* __restrict__ heat, int H, int W, int tiles_x, int max_peaks, float thr, int vec,
                 u64* __restrict__ ws_keys, int* __restrict__ ws_count) {
  using T = PeakTile<R>;
  extern __shared__ __align__(16) unsigned char smem[];
  u64* keys = reinterpret_cast<u64*>(smem + T::keys_off);
  float* raw = reinterpret_cast<float*>(smem + T::raw_off);
  float* mrow = reinterpret_cast<float*>(smem + T::mrow_off);
  uint8_t* flag = smem + T::flag_off;
  __shared__ int s_count;

  const int map = blockIdx.y, tile = blockIdx.x;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int y0 = ty * kPeakTH, x0 = tx * kPeakTW;
  const int gy0 = y0 - R, gx0 = x0 - T::R4;              // image coordinates of raw[0][0]
  const float* src = heat + (size_t)map * H * W;
  const int tid = threadIdx.x;
  const size_t slot = (size_t)map * gridDim.x + tile;
  if (tid == 0) s_count = 0;

  // ---- 1. haloed tile -> raw (outside the image and NaN -> -inf); four loads in flight per thread
  bool any = false;   // some pixel of the output tile reaches the threshold
  if (vec) {          // W % 4 == 0 and a 16-byte aligned map: every float4 lies wholly inside or wholly outside the image
    constexpr int qrow = T::pitch / 4, nq = T::rows * qrow;
    for (int base = tid; base < nq; base += 4 * kPeakThreads) {
      float4 q[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * kPeakThreads;
        const int row = i / qrow, gy = gy0 + row, gx = gx0 + 4 * (i - row * qrow);
        q[u] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
        if (i < nq && gy >= 0 && gy < H && gx >= 0 && gx < W) q[u] = __ldg(reinterpret_cast<const float4*>(src + (size_t)gy * W + gx));
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * kPeakThreads;
        if (i < nq) {
          const int row = i / qrow, c = 4 * (i - row * qrow);
          const float4 v = make_float4(nan_to_ninf(q[u].x), nan_to_ninf(q[u].y), nan_to_ninf(q[u].z), nan_to_ninf(q[u].w));
          reinterpret_cast<float4*>(raw + row * T::pitch)[c >> 2] = v;
          if (row >= R && row < R + kPeakTH && c >= T::R4 && c < T::R4 + kPeakTW)
            any |= v.x >= thr || v.y >= thr || v.z >= thr || v.w >= thr;
        }
      }
    }
  } else {
    constexpr int n = T::rows * T::pitch;
    for (int base = tid; base < n; base += 4 * kPeakThreads) {
      float q[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * kPeakThreads;
        const int row = i / T::pitch, gy = gy0 + row, gx = gx0 + (i - row * T::pitch);
        q[u] = -INFINITY;
        if (i < n && gy >= 0 && gy < H && gx >= 0 && gx < W) q[u] = __ldg(src + (size_t)gy * W + gx);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * kPeakThreads;
        if (i < n) {
          const int row = i / T::pitch, c = i - row * T::pitch;
          const float v = nan_to_ninf(q[u]);
          raw[i] = v;
          if (row >= R && row < R + kPeakTH && c >= T::R4 && c < T::R4 + kPeakTW) any |= v >= thr;
        }
      }
    }
  }
  if (!__syncthreads_or(any)) {   // nothing reaches the threshold (the common case on a sigmoid heatmap): no peaks here
    if (tid == 0) ws_count[slot] = 0;
    return;
  }

  // ---- 2. rows pass: Mrow of every halo row; for the tile's rows also the row half of the test -> flag
  constexpr int runs = kPeakTW / kPeakRowRun;
  constexpr int nv = kPeakRowRun + 2 * T::R4;
  for (int item = tid; item < T::rows * runs; item += kPeakThreads) {
    const int row = item / runs, c0 = (item - row * runs) * kPeakRowRun;
    float v[nv];
    const float4* rp = reinterpret_cast<const float4*>(raw + row * T::pitch + c0);
#pragma unroll
    for (int j = 0; j < nv / 4; ++j) {
      const float4 q = rp[j];
      v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
    }
    float m[kPeakRowRun];
#pragma unroll
    for (int j = 0; j < kPeakRowRun; ++j) {
      float mx = v[T::R4 + j];
#pragma unroll
      for (int d = 1; d <= R; ++d) mx = fmaxf(mx, fmaxf(v[T::R4 + j - d], v[T::R4 + j + d]));
      m[j] = mx;
    }
    float4* mp = reinterpret_cast<float4*>(mrow + row * kPeakTW + c0);
#pragma unroll
    for (int j = 0; j < kPeakRowRun / 4; ++j) mp[j] = make_float4(m[4 * j], m[4 * j + 1], m[4 * j + 2], m[4 * j + 3]);
    if (row >= R && row < R + kPeakTH) {
      uint32_t f[2] = {0u, 0u};
#pragma unroll
      for (int j = 0; j < kPeakRowRun; ++j) {
        const float p = v[T::R4 + j];
        float l = v[T::R4 + j - 1];
#pragma unroll
        for (int d = 2; d <= R; ++d) l = fmaxf(l, v[T::R4 + j - d]);
        if (p >= thr && p >= m[j] && p > l) f[j >> 2] |= 1u << (8 * (j & 3));
      }
      *reinterpret_cast<uint2*>(flag + (row - R) * kPeakTW + c0) = make_uint2(f[0], f[1]);
    }
  }
  __syncthreads();

  // ---- 3. columns pass: U and Dn for the flagged pixels; every peak appends its key
  {
    const int c = tid % kPeakTW, r0 = (tid / kPeakTW) * kPeakColRun;
    float m[kPeakColRun + 2 * R];   // Mrow of halo rows r0 .. r0 + kPeakColRun + 2R - 1 (tile row t = halo row t + R)
#pragma unroll
    for (int k = 0; k < kPeakColRun + 2 * R; ++k) m[k] = mrow[(r0 + k) * kPeakTW + c];
#pragma unroll
    for (int i = 0; i < kPeakColRun; ++i) {
      if (flag[(r0 + i) * kPeakTW + c]) {
        const float p = raw[(r0 + i + R) * T::pitch + T::R4 + c];
        float up = m[i], dn = m[i + R];
#pragma unroll
        for (int d = 1; d < R; ++d) up = fmaxf(up, m[i + d]);
#pragma unroll
        for (int d = 1; d <= R; ++d) dn = fmaxf(dn, m[i + R + d]);
        if (p >= dn && p > up) {
          const uint32_t idx = (uint32_t)(y0 + r0 + i) * (uint32_t)W + (uint32_t)(x0 + c);
          keys[atomicAdd(&s_count, 1)] = ((u64)peak_orderable(p) << 32) | (u64)(~idx);
        }
      }
    }
  }
  __syncthreads();

  // ---- 4. sort the tile's keys (descending) and keep the top N
  const int n = s_count;
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = n + tid; i < P; i += kPeakThreads) keys[i] = 0ull;   // below every key (a key's high word is >= orderable(-inf) > 0)
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < P; i += kPeakThreads) {
        const int l = i ^ j;
        if (l > i) {
          const u64 a = keys[i], b = keys[l];
          if (((i & k) == 0) ? a < b : a > b) {
            keys[i] = b;
            keys[l] = a;
          }
        }
      }
      __syncthreads();
    }
  }
  const int keep = min(n, max_peaks);
  for (int i = tid; i < keep; i += kPeakThreads) ws_keys[slot * max_peaks + i] = keys[i];
  if (tid == 0) ws_count[slot] = keep;
}

// lists merged per round: their filled slots are loaded together (one round trip), then folded into the running top N one by one
constexpr int kMergeKeys = 4096, kMergeMaxLists = 1024;

// number of entries of the descending list s[0..n) that are greater than key
__device__ __forceinline__ int rank_in(const u64* s, int n, u64 key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (s[mid] > key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(kPeakThreads)
peak_merge_kernel(const u64* __restrict__ ws_keys, const int* __restrict__ ws_count, int tiles, int N, int W, int32_t* __restrict__ yx,
                  float* __restrict__ score, int32_t* __restrict__ count) {
  __shared__ u64 top[2][kPeakMaxN];
  __shared__ u64 lists[kMergeKeys];
  __shared__ int cnt[kMergeMaxLists];
  const int map = blockIdx.x, tid = threadIdx.x;
  const u64* mk = ws_keys + (size_t)map * tiles * N;
  const int* mc = ws_count + (size_t)map * tiles;
  const int G = min(kMergeKeys / N, kMergeMaxLists);
  int a = 0, cur = 0;
  for (int t0 = 0; t0 < tiles; t0 += G) {
    const int g = min(G, tiles - t0);
    for (int i = tid; i < g; i += kPeakThreads) cnt[i] = mc[t0 + i];
    __syncthreads();
    for (int i = tid; i < g * N; i += kPeakThreads) {
      const int l = i / N;
      if (i - l * N < cnt[l]) lists[i] = mk[(size_t)t0 * N + i];
    }
    __syncthreads();
    for (int l = 0; l < g; ++l) {
      const int b = cnt[l];
      const u64* B = lists + l * N;
      if (b == 0 || (a == N && B[0] < top[cur][N - 1])) continue;   // block-uniform: nothing of this list enters the top N
      const u64* A = top[cur];
      u64* O = top[cur ^ 1];
      for (int i = tid; i < a; i += kPeakThreads) {
        const int pos = i + rank_in(B, b, A[i]);
        if (pos < N) O[pos] = A[i];
      }
      for (int i = tid; i < b; i += kPeakThreads) {
        const int pos = i + rank_in(A, a, B[i]);
        if (pos < N) O[pos] = B[i];
      }
      __syncthreads();
      a = min(N, a + b);
      cur ^= 1;
    }
    __syncthreads();   // cnt / lists are refilled next round
  }
  for (int i = tid; i < N; i += kPeakThreads) {
    const size_t o = (size_t)map * N + i;
    if (i < a) {
      const u64 k = top[cur][i];
      const uint32_t idx = ~(uint32_t)k;
      yx[2 * o] = (int32_t)(idx / (uint32_t)W);
      yx[2 * o + 1] = (int32_t)(idx % (uint32_t)W);
      score[o] = peak_value((uint32_t)(k >> 32));
    } else {
      yx[2 * o] = -1;
      yx[2 * o + 1] = -1;
      score[o] = -INFINITY;
    }
  }
  if (tid == 0) count[map] = a;
}

static int peak_tiles(int H, int W, int* tiles_x) {
  *tiles_x = ceil_div(W, kPeakTW);
  return ceil_div(H, kPeakTH) * *tiles_x;
}

template <int R>
static int launch_peak_tile(dim3 grid, cudaStream_t s, const float* heat, int H, int W, int tiles_x, int N, float thr, int vec,
                            u64* keys, int* cnt) {
  if (int rc = opt_in_smem<peak_tile_kernel<R>>(PeakTile<R>::bytes, "hk_peak_decode")) return rc;
  peak_tile_kernel<R><<<grid, kPeakThreads, PeakTile<R>::bytes, s>>>(heat, H, W, tiles_x, N, thr, vec, keys, cnt);
  return check_launch("peak_tile_kernel");
}

typedef int (*PeakTileLaunch)(dim3, cudaStream_t, const float*, int, int, int, int, float, int, u64*, int*);
static const PeakTileLaunch kPeakTileLaunch[kPeakMaxR] = {
    launch_peak_tile<1>,  launch_peak_tile<2>,  launch_peak_tile<3>,  launch_peak_tile<4>,  launch_peak_tile<5>,  launch_peak_tile<6>,
    launch_peak_tile<7>,  launch_peak_tile<8>,  launch_peak_tile<9>,  launch_peak_tile<10>, launch_peak_tile<11>, launch_peak_tile<12>,
    launch_peak_tile<13>, launch_peak_tile<14>, launch_peak_tile<15>, launch_peak_tile<16>};

}  // namespace hk

extern "C" {

size_t hk_peak_workspace_bytes(int B, int K, int H, int W, int max_peaks, int min_distance) {
  if (B <= 0 || K <= 0 || H <= 0 || W <= 0 || max_peaks < 1 || max_peaks > hk::kPeakMaxN || min_distance < 1 ||
      min_distance > hk::kPeakMaxR)
    return 0;
  int tiles_x;
  const size_t slots = (size_t)B * K * hk::peak_tiles(H, W, &tiles_x);
  return slots * max_peaks * sizeof(hk::u64) + slots * sizeof(int);   // sorted keys per tile, then the count per tile
}

int hk_peak_decode(const float* heat, int B, int K, int H, int W, int max_peaks, int min_distance, float threshold, int32_t* yx,
                   float* score, int32_t* count, void* ws, size_t ws_bytes, void* stream) {
  using namespace hk;
  HK_REQUIRE(heat && yx && score && count && ws, "hk_peak_decode: null pointer");
  HK_REQUIRE(B > 0 && K > 0 && H > 0 && W > 0, "hk_peak_decode: bad shape B=%d K=%d H=%d W=%d", B, K, H, W);
  HK_REQUIRE((long long)H * W < 0x7fffffffLL, "hk_peak_decode: map too large");
  HK_REQUIRE((long long)B * K <= 65535, "hk_peak_decode: B*K=%lld exceeds grid.y", (long long)B * K);
  HK_REQUIRE(max_peaks >= 1 && max_peaks <= kPeakMaxN, "hk_peak_decode: max_peaks=%d outside [1, %d]", max_peaks, kPeakMaxN);
  HK_REQUIRE(min_distance >= 1 && min_distance <= kPeakMaxR, "hk_peak_decode: min_distance=%d outside [1, %d]", min_distance, kPeakMaxR);
  HK_REQUIRE(isfinite(threshold), "hk_peak_decode: threshold must be finite");
  HK_REQUIRE(ws_bytes >= hk_peak_workspace_bytes(B, K, H, W, max_peaks, min_distance), "hk_peak_decode: workspace too small");
  HK_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7) == 0, "hk_peak_decode: workspace must be 8-byte aligned");
  int tiles_x;
  const int tiles = peak_tiles(H, W, &tiles_x);
  const int maps = B * K;
  u64* keys = static_cast<u64*>(ws);
  int* cnt = reinterpret_cast<int*>(keys + (size_t)maps * tiles * max_peaks);
  const int vec = (W % 4 == 0) && (reinterpret_cast<uintptr_t>(heat) & 15) == 0;
  cudaStream_t s = as_stream(stream);
  int rc = kPeakTileLaunch[min_distance - 1](dim3(tiles, maps), s, heat, H, W, tiles_x, max_peaks, threshold, vec, keys, cnt);
  if (rc) return rc;
  peak_merge_kernel<<<maps, kPeakThreads, 0, s>>>(keys, cnt, tiles, max_peaks, W, yx, score, count);
  return check_launch("peak_merge_kernel");
}

}  // extern "C"
