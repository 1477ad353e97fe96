// Per-pixel confidence of the disparity from the classif head's distribution over disparity (gwcnet_dca_g.py:235-239):
// p = softmax_d(logits), peak_q = max_d p, std_q = sqrt(sum_d p(d) (d - mu)^2) with mu = sum_d d p(d) (= pred_quarter),
// both convex-upsampled x4 with the prop net's 9-neighbour weights exactly as pred4 is (convex_upsample_kernel,
// gwcnet_dca_g.py:117-124): peak = up(peak_q), std = up(4 std_q).  Definitions: include/dca_b200.h section (4).
//
// Same tiling as softmax_regress_upsample_kernel (dca_ops.cu): a CTA owns a 32 x 8 tile of 1/4-res pixels, computes the
// two statistics of the tile and its 1-pixel ring (recomputed by the neighbouring CTAs; zero outside the image, the
// zero padding of F.unfold) into shared memory, writes the tile's own 1/4-res values, then upsamples both channels from
// shared memory with one read of each mask float4.
#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int CF_TW = 32, CF_TH = 8;

// max, then sum and mean exactly as softmax_regress_kernel forms them, then the centred second moment: a third pass over
// the (L1-resident) logits instead of E[d^2] - mu^2, which cancels catastrophically on confident pixels
__device__ __forceinline__ void pixel_confidence(const float* __restrict__ lp, size_t HW, int D, float& peak, float& sd) {
  float m = -INFINITY;
  for (int d = 0; d < D; ++d) m = fmaxf(m, lp[(size_t)d * HW]);
  float sum = 0.f, acc = 0.f;
  for (int d = 0; d < D; ++d) {
    const float ev = expf(lp[(size_t)d * HW] - m);
    sum += ev;
    acc = fmaf(ev, (float)d, acc);
  }
  const float mu = acc / sum;
  float var = 0.f;
  for (int d = 0; d < D; ++d) {
    const float ev = expf(lp[(size_t)d * HW] - m);
    const float c = (float)d - mu;
    var = fmaf(ev * c, c, var);
  }
  peak = 1.f / sum;                 // p(argmax) = exp(m - m) / sum
  sd = sqrtf(var / sum);
}

__global__ void __launch_bounds__(CF_TW * CF_TH)
softmax_confidence_upsample_kernel(const float* __restrict__ logits, const float* __restrict__ mask,
                                   float* __restrict__ peak_q, float* __restrict__ std_q, float* __restrict__ peak,
                                   float* __restrict__ stdv, int B, int D, int H, int W) {
  __shared__ float s_pk[CF_TH + 2][CF_TW + 2];
  __shared__ float s_sd[CF_TH + 2][CF_TW + 2];
  const int b = blockIdx.z, h0 = blockIdx.y * CF_TH, w0 = blockIdx.x * CF_TW;
  const size_t HW = (size_t)H * W;
  pdl_wait();
  for (int i = threadIdx.x; i < (CF_TH + 2) * (CF_TW + 2); i += blockDim.x) {
    const int ly = i / (CF_TW + 2), lx = i - ly * (CF_TW + 2);
    const int h = h0 + ly - 1, w = w0 + lx - 1;
    float pk = 0.f, sd = 0.f;
    if (h >= 0 && h < H && w >= 0 && w < W) {
      pixel_confidence(logits + (size_t)b * D * HW + (size_t)h * W + w, HW, D, pk, sd);
      if (ly >= 1 && ly <= CF_TH && lx >= 1 && lx <= CF_TW) {
        const size_t o = (size_t)b * HW + (size_t)h * W + w;
        if (peak_q) peak_q[o] = pk;
        if (std_q) std_q[o] = sd;
      }
    }
    s_pk[ly][lx] = pk;
    s_sd[ly][lx] = sd;
  }
  __syncthreads();
  for (int it = threadIdx.x; it < CF_TW * CF_TH * 4; it += blockDim.x) {
    const int i = it & 3, px = it >> 2;
    const int lx = px % CF_TW, ly = px / CF_TW;
    const int h = h0 + ly, w = w0 + lx;
    if (h >= H || w >= W) continue;
    const float* mp = mask + (((size_t)b * H + h) * W + w) * 144 + i * 4;
    float4 mv[9];
#pragma unroll
    for (int n = 0; n < 9; ++n) mv[n] = *reinterpret_cast<const float4*>(mp + n * 16);
    float4 mx = mv[0];
#pragma unroll
    for (int n = 1; n < 9; ++n) {
      mx.x = fmaxf(mx.x, mv[n].x); mx.y = fmaxf(mx.y, mv[n].y); mx.z = fmaxf(mx.z, mv[n].z); mx.w = fmaxf(mx.w, mv[n].w);
    }
    float4 sm = make_float4(0, 0, 0, 0), ap = make_float4(0, 0, 0, 0), as = make_float4(0, 0, 0, 0);
#pragma unroll
    for (int n = 0; n < 9; ++n) {
      const float pv = s_pk[ly + n / 3][lx + n % 3], sv = 4.f * s_sd[ly + n / 3][lx + n % 3];
      const float ex = expf(mv[n].x - mx.x), ey = expf(mv[n].y - mx.y), ez = expf(mv[n].z - mx.z),
                  ew = expf(mv[n].w - mx.w);
      sm.x += ex; sm.y += ey; sm.z += ez; sm.w += ew;
      ap.x = fmaf(ex, pv, ap.x); ap.y = fmaf(ey, pv, ap.y); ap.z = fmaf(ez, pv, ap.z); ap.w = fmaf(ew, pv, ap.w);
      as.x = fmaf(ex, sv, as.x); as.y = fmaf(ey, sv, as.y); as.z = fmaf(ez, sv, as.z); as.w = fmaf(ew, sv, as.w);
    }
    const size_t o = ((size_t)b * 4 * H + 4 * h + i) * (4 * W) + 4 * w;
    *reinterpret_cast<float4*>(peak + o) = make_float4(ap.x / sm.x, ap.y / sm.y, ap.z / sm.z, ap.w / sm.w);
    *reinterpret_cast<float4*>(stdv + o) = make_float4(as.x / sm.x, as.y / sm.y, as.z / sm.z, as.w / sm.w);
  }
}

}  // namespace dca

using namespace dca;

extern "C" int dca_softmax_confidence_upsample(const float* logits, const float* mask, float* peak_q, float* std_q,
                                               float* peak, float* std, int B, int D, int H, int W, void* stream) {
  if (!logits || !mask || !peak || !std || B <= 0 || D <= 0 || H <= 0 || W <= 0 || B > 65535) return DCA_ERR_ARG;
  dca_launch(softmax_confidence_upsample_kernel, dim3((W + CF_TW - 1) / CF_TW, (H + CF_TH - 1) / CF_TH, B),
             CF_TW * CF_TH, 0, (cudaStream_t)stream, logits, mask, peak_q, std_q, peak, std, B, D, H, W);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
