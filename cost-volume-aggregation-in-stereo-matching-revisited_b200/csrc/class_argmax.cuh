// Per-pixel softmax / first-argmax over the disparity classes of fp32 logits, shared by dca_class_stats (dca_ops.cu) and
// dca_class_confusion (metrics.cu): both must pick the same class for every pixel, bit for bit.
#pragma once
#include "dca_common.cuh"

namespace dca {

constexpr int CS_G = 8;                      // class groups per pixel: thread (lane = pixel, group g) owns classes g, g + 8, ...
constexpr int CS_PER = 8;                    // ... up to 8 of them in registers (D <= 64; more: they are re-read)
constexpr int CS_THREADS = 32 * CS_G;

// Per-pixel class statistics by a (32 pixels x CS_G groups) thread block.  A single thread per pixel ran 3,500 dependent
// instructions (24 x (expf + expf + divide)) on a warp that had its scheduler to itself: 17 us for 7,488 pixels.  Here the
// classes of a pixel are dealt out over CS_G threads (same lane, different warps: loads stay coalesced along w) and the
// max / sum / first-argmax are merged through shared memory in a FIXED order, so the result is still reproducible bit
// for bit.  P[d] = exp(x[d] - m) / s with m = max_d x[d], s = sum_d exp(x[d] - m) (groups summed in the order 0..7);
// strict > inside a thread (ascending d) and "larger P, then smaller d" across threads keep torch.argmax's FIRST maximum.
// `load(d)` returns the pixel's logit d; all CS_THREADS threads must call this (it synchronises); valid = the lane
// holds a pixel.  Returns k (class) and e = exp(P[k]) to the threads with g == 0.
struct CsSmem { float red[CS_G][32]; int idx[CS_G][32]; };
// BAR = 0: the whole block takes part (__syncthreads); BAR > 0: only the first CS_THREADS threads do (named barrier BAR)
template <int BAR>
__device__ __forceinline__ void cs_sync() {
  if (BAR == 0) __syncthreads();
  else asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(CS_THREADS) : "memory");
}
template <int BAR, typename Load>
__device__ __forceinline__ void pixel_class_stats(CsSmem& sm, int lane, int g, int D, bool valid, Load load, int& k_out,
                                                  float& e_out) {
  float v[CS_PER];
  float m = -INFINITY;
  if (valid) {
#pragma unroll
    for (int i = 0; i < CS_PER; ++i) {
      const int d = g + CS_G * i;
      v[i] = d < D ? load(d) : -INFINITY;
      m = fmaxf(m, v[i]);
    }
    for (int d = g + CS_G * CS_PER; d < D; d += CS_G) m = fmaxf(m, load(d));
  }
  sm.red[g][lane] = m;
  cs_sync<BAR>();
#pragma unroll
  for (int j = 0; j < CS_G; ++j) m = fmaxf(m, sm.red[j][lane]);
  cs_sync<BAR>();
  float s = 0.f;
  if (valid) {
#pragma unroll
    for (int i = 0; i < CS_PER; ++i) {
      const int d = g + CS_G * i;
      v[i] = d < D ? expf(v[i] - m) : 0.f;
      s += v[i];
    }
    for (int d = g + CS_G * CS_PER; d < D; d += CS_G) s += expf(load(d) - m);
  }
  sm.red[g][lane] = s;
  cs_sync<BAR>();
  s = 0.f;
#pragma unroll
  for (int j = 0; j < CS_G; ++j) s += sm.red[j][lane];
  cs_sync<BAR>();
  float best = -1.f;
  int k = 0;
  if (valid) {
#pragma unroll
    for (int i = 0; i < CS_PER; ++i) {
      const int d = g + CS_G * i;
      const float pd = v[i] / s;                        // same formula torch's softmax uses
      if (d < D && pd > best) { best = pd; k = d; }     // ascending d, strict >: the first maximum of this thread
    }
    for (int d = g + CS_G * CS_PER; d < D; d += CS_G) {
      const float pd = expf(load(d) - m) / s;
      if (pd > best) { best = pd; k = d; }
    }
  }
  sm.red[g][lane] = best;
  sm.idx[g][lane] = k;
  cs_sync<BAR>();
  if (g == 0) {
#pragma unroll
    for (int j = 1; j < CS_G; ++j) {
      const float bj = sm.red[j][lane];
      const int kj = sm.idx[j][lane];
      if (bj > best || (bj == best && kj < k)) { best = bj; k = kj; }
    }
    k_out = k;
    e_out = expf(best);
  }
}

}  // namespace dca
