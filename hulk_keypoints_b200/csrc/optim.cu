// Fused Adam over flat fp32 buffers (SURVEY.md §8 f2).  Replaces the ~220 small launches per step of
// torch.optim.Adam(lr=1e-4, weight_decay=1e-4) at reference train.py:79,36 with one HBM-bound pass:
// 16 B read + 12 B written per parameter (p, g, m, v in; p, m, v out), 21.8 M parameters -> 0.61 GB per step.
// Arithmetic follows torch's single-tensor Adam (no amsgrad) operation by operation:
//   coupled L2:  g += wd*p
//   decoupled:   p *= 1 - lr*wd                       (torch.optim.AdamW / Adam(decoupled_weight_decay=True))
//   then         m += (g-m)*(1-b1);  v = v*b2 + (1-b2)*g*g;  p -= (lr/(1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
// Hyperparameters and bias corrections come from a table of segments (runs of the flat buffer that share them, in float4 units),
// passed by value as a __grid_constant__ launch parameter: one launch per step whatever the number of parameter groups.
#include "hk_common.cuh"

namespace hk {

template <int CAP>
struct AdamTable {
  HkAdamSegment seg[CAP];
};

// Each CTA updates one contiguous chunk of float4s and looks up the segment of its first element once; its threads then walk the
// (sorted, contiguous) table forward as their index crosses a segment end -- no per-element search, no global-memory table.
template <int CAP>
__global__ void __launch_bounds__(256)
adam_segments_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n4,
                     long long n, long long chunk, int nseg, const __grid_constant__ AdamTable<CAP> t) {
  const long long lo = (long long)blockIdx.x * chunk;
  const long long hi = lo + chunk < n4 ? lo + chunk : n4;
  int s = 0;
  for (int b = nseg - 1; s < b;) {   // first segment ending past lo
    const int mid = (s + b) >> 1;
    if (t.seg[mid].end4 > lo) b = mid; else s = mid + 1;
  }
  for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    while (i >= t.seg[s].end4) ++s;
    const HkAdamSegment& sg = t.seg[s];
    const float lr_over_bc1 = sg.lr_over_bc1, inv_sqrt_bc2 = sg.inv_sqrt_bc2, b1 = sg.beta1, b2 = sg.beta2, eps = sg.eps;
    const float wd = sg.weight_decay, decay = sg.decay;
    const bool decoupled = sg.decoupled != 0;
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = __ldcs(reinterpret_cast<const float4*>(g) + i);
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pa = reinterpret_cast<float*>(&pp);
    const float* ga = reinterpret_cast<const float*>(&gg);
    float* ma = reinterpret_cast<float*>(&mm);
    float* va = reinterpret_cast<float*>(&vv);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float pj = pa[j], grad;
      if (decoupled) {
        pj = __fmul_rn(pj, decay);   // its own rounding, as torch's param.mul_(1 - lr*wd)
        grad = ga[j];
      } else {
        grad = fmaf(wd, pj, ga[j]);
      }
      ma[j] = fmaf(grad - ma[j], 1.0f - b1, ma[j]);
      va[j] = fmaf(va[j], b2, (1.0f - b2) * grad * grad);
      const float denom = fmaf(sqrtf(va[j]), inv_sqrt_bc2, eps);
      pa[j] = pj - lr_over_bc1 * (ma[j] / denom);
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  // scalar tail (n % 4): the partial float4 at index n4 belongs to the last segment
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const HkAdamSegment& sg = t.seg[nseg - 1];
    const float lr_over_bc1 = sg.lr_over_bc1, inv_sqrt_bc2 = sg.inv_sqrt_bc2, b1 = sg.beta1, b2 = sg.beta2, eps = sg.eps;
    const long long i = (n4 << 2) + threadIdx.x;
    float pi = p[i], grad;
    if (sg.decoupled) {
      pi = __fmul_rn(pi, sg.decay);
      grad = g[i];
    } else {
      grad = fmaf(sg.weight_decay, pi, g[i]);
    }
    const float mi = fmaf(grad - m[i], 1.0f - b1, m[i]);
    const float vi = fmaf(v[i], b2, (1.0f - b2) * grad * grad);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi - lr_over_bc1 * (mi / fmaf(sqrtf(vi), inv_sqrt_bc2, eps));
  }
}

template <int CAP>
int launch_adam_segments(float* p, const float* g, float* m, float* v, long long n, const HkAdamSegment* segs, int nseg,
                         cudaStream_t stream) {
  AdamTable<CAP> t;
  for (int k = 0; k < nseg; ++k) t.seg[k] = segs[k];
  const long long n4 = n >> 2;
  const long long work = n4 > 0 ? n4 : 1;
  long long blocks = ceil_div_ll(work, 256);
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  const long long chunk = ceil_div_ll(ceil_div_ll(work, blocks), 256) * 256;   // whole 256-thread sweeps per CTA
  blocks = ceil_div_ll(work, chunk);
  adam_segments_kernel<CAP><<<(int)blocks, 256, 0, stream>>>(p, g, m, v, n4, n, chunk, nseg, t);
  return check_launch("adam_segments_kernel");
}

}  // namespace hk

extern "C" int hk_adam_step_segments(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n,
                                     const HkAdamSegment* segments, int num_segments, void* stream) {
  using namespace hk;
  HK_REQUIRE(params && grads && exp_avg && exp_avg_sq && segments, "hk_adam_step_segments: null pointer");
  HK_REQUIRE(n > 0, "hk_adam_step_segments: n must be positive");
  HK_REQUIRE(num_segments >= 1 && num_segments <= HK_ADAM_MAX_SEGMENTS,
             "hk_adam_step_segments: %d segments, the table holds 1..%d (a launch parameter of at most 32 KB)", num_segments,
             HK_ADAM_MAX_SEGMENTS);
  HK_REQUIRE(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(exp_avg) |
               reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0, "hk_adam_step_segments: buffers must be 16-byte aligned");
  long long at = 0;
  for (int k = 0; k < num_segments; ++k) {
    HK_REQUIRE(segments[k].begin4 == at && segments[k].end4 > at,
               "hk_adam_step_segments: segment %d is [%lld, %lld); segments must be non-empty, sorted and contiguous from 0", k,
               segments[k].begin4, segments[k].end4);
    at = segments[k].end4;
  }
  HK_REQUIRE(at == ceil_div_ll(n, 4), "hk_adam_step_segments: the segments cover %lld float4s, n = %lld needs %lld", at, n,
             ceil_div_ll(n, 4));
  if (num_segments <= 8) return launch_adam_segments<8>(params, grads, exp_avg, exp_avg_sq, n, segments, num_segments, as_stream(stream));
  return launch_adam_segments<HK_ADAM_MAX_SEGMENTS>(params, grads, exp_avg, exp_avg_sq, n, segments, num_segments, as_stream(stream));
}

extern "C" int hk_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                            float beta1, float beta2, float eps, float weight_decay, int step, void* stream) {
  HK_REQUIRE(n > 0 && step >= 1, "hk_adam_step: n and step must be positive");
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  HkAdamSegment seg = {};
  seg.begin4 = 0;
  seg.end4 = (n + 3) / 4;
  seg.lr_over_bc1 = (float)((double)lr / bc1);
  seg.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  seg.beta1 = beta1;
  seg.beta2 = beta2;
  seg.eps = eps;
  seg.weight_decay = weight_decay;
  seg.decay = 1.0f;
  seg.decoupled = 0;
  return hk_adam_step_segments(params, grads, exp_avg, exp_avg_sq, n, &seg, 1, stream);
}
