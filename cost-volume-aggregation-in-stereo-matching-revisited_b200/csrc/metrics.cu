// Accuracy against ground-truth disparity: the scoring half of the reference's evaluation loop (main_dca.py `mytest`
// :143-232; EPE / N-px error / D1 formulas of utils/metrics.py:45-63, the class-map confusion matrix of the segmentation
// Evaluator :66-120).  Counters are 64-bit integers ADDED into caller-owned tables, so results do not depend on the
// order in which blocks arrive and a CUDA graph can capture both launches.
//
//   disparity_metrics   per image: valid / sum |pred - gt| (fixed point) / E > 1, 2, 3 / D1 / non-finite predictions
//   class_confusion     conf[gt class][predicted class] of the 1/8-res DCA class maps
//   confidence_histograms  (count, sum |E|) per confidence bin and per error bin: the sparsification curves
//   depth_metrics       per image: the depth errors of the Eigen et al. protocol from disparities and one calibration
#include <limits.h>

#include "dca_common.cuh"
#include "class_argmax.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int MT_THREADS = 256;
constexpr int MT_WARPS = MT_THREADS / 32;
constexpr float MT_FIX = 1048576.0f;      // 2^20: SUM_ABS unit is 2^-20 px
constexpr float MT_CLAMP = 1048576.0f;    // E is clamped to 2^20 px before scaling: <= 2^40 per pixel

__device__ __forceinline__ bool gt_valid(float g, float max_valid) {
  return isfinite(g) && g > 0.f && (max_valid <= 0.f || g < max_valid);
}

struct MetricAcc {
  unsigned valid, gt1, gt2, gt3, d1, nonfinite;
  unsigned long long sum;
};

// |E| in the fixed point of DCA_METRIC_SUM_ABS (2^-20 px units)
__device__ __forceinline__ unsigned long long abs_err_fix(float e) {
  return __float2ull_rn(__fmul_rn(fminf(e, MT_CLAMP), MT_FIX));
}

__device__ __forceinline__ void metric_pixel(float p, float g, float max_valid, MetricAcc& a) {
  if (!gt_valid(g, max_valid)) return;
  const float e = fabsf(__fsub_rn(p, g));
  const bool bad = !isfinite(p);               // NaN / inf prediction: an error of every kind, kept out of the sum
  a.valid += 1;
  a.nonfinite += bad;
  if (!bad) a.sum += abs_err_fix(e);
  a.gt1 += bad || e > 1.f;
  a.gt2 += bad || e > 2.f;
  a.gt3 += bad || e > 3.f;
  a.d1 += bad || (e > 3.f && __fdiv_rn(e, fabsf(g)) > 0.05f);
}

// grid (blocks per image, B); every block adds its totals with one atomic per (image, counter)
__global__ void __launch_bounds__(MT_THREADS)
disparity_metrics_kernel(const float* __restrict__ pred, const float* __restrict__ gt, unsigned long long* __restrict__ rows,
                         int HW, int vec4, float max_valid) {
  __shared__ unsigned long long red[MT_WARPS][DCA_METRIC_COUNT];
  pdl_wait();
  const int b = blockIdx.y;
  const float* pb = pred + (size_t)b * HW;
  const float* gb = gt + (size_t)b * HW;
  MetricAcc a = {0u, 0u, 0u, 0u, 0u, 0u, 0ull};
  const int stride = gridDim.x * blockDim.x;
  if (vec4) {
    const float4* p4 = reinterpret_cast<const float4*>(pb);
    const float4* g4 = reinterpret_cast<const float4*>(gb);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW / 4; i += stride) {
      const float4 p = __ldg(p4 + i), g = __ldg(g4 + i);
      metric_pixel(p.x, g.x, max_valid, a);
      metric_pixel(p.y, g.y, max_valid, a);
      metric_pixel(p.z, g.z, max_valid, a);
      metric_pixel(p.w, g.w, max_valid, a);
    }
  } else {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += stride)
      metric_pixel(__ldg(pb + i), __ldg(gb + i), max_valid, a);
  }
  const unsigned full = 0xffffffffu;
  unsigned long long v[DCA_METRIC_COUNT];
  v[DCA_METRIC_VALID] = __reduce_add_sync(full, a.valid);
  v[DCA_METRIC_GT1] = __reduce_add_sync(full, a.gt1);
  v[DCA_METRIC_GT2] = __reduce_add_sync(full, a.gt2);
  v[DCA_METRIC_GT3] = __reduce_add_sync(full, a.gt3);
  v[DCA_METRIC_D1] = __reduce_add_sync(full, a.d1);
  v[DCA_METRIC_PRED_NONFINITE] = __reduce_add_sync(full, a.nonfinite);
  unsigned long long s = a.sum;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(full, s, o);
  v[DCA_METRIC_SUM_ABS] = s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int m = 0; m < DCA_METRIC_COUNT; ++m) red[warp][m] = v[m];
  }
  __syncthreads();
  if (threadIdx.x < DCA_METRIC_COUNT) {
    unsigned long long t = 0;
#pragma unroll
    for (int w = 0; w < MT_WARPS; ++w) t += red[w][threadIdx.x];
    if (t) atomicAdd(rows + (size_t)b * DCA_METRIC_COUNT + threadIdx.x, t);
  }
}

// One 32-pixel run of a 1/8-res row segment per iteration, its classes dealt out over the CS_G warps of the block by
// pixel_class_stats (the routine of dca_class_stats, so both pick the same class bit for bit); counts go to a
// shared-memory histogram [D][D], flushed with one global atomic per non-zero bin.
__global__ void __launch_bounds__(CS_THREADS)
class_confusion_kernel(const float* __restrict__ logits, const float* __restrict__ gt, unsigned long long* __restrict__ conf,
                       int B, int D, int H8, int W8, float max_valid) {
  extern __shared__ unsigned hist[];
  __shared__ CsSmem sm;
  for (int i = threadIdx.x; i < D * D; i += CS_THREADS) hist[i] = 0u;
  pdl_wait();
  __syncthreads();
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int HW = H8 * W8, chunks = (HW + 31) / 32;
  const size_t W = (size_t)8 * W8;
  for (int c = blockIdx.x; c < B * chunks; c += gridDim.x) {     // uniform over the block: pixel_class_stats syncs
    const int b = c / chunks, p = (c - b * chunks) * 32 + lane;
    int gcls = -1;
    if (p < HW) {
      const int i = p / W8, j = p - i * W8;
      const float gv = __ldg(gt + ((size_t)b * 8 * H8 + 8 * i) * W + 8 * j);
      if (gt_valid(gv, max_valid))
        gcls = (int)fminf(floorf(__fadd_rn(__fmul_rn(gv, 0.125f), 0.5f)), (float)(D - 1));
    }
    const float* lp = logits + (size_t)b * D * HW + (gcls >= 0 ? p : 0);
    int k = 0;
    float e = 0.f;
    pixel_class_stats<0>(sm, lane, g, D, gcls >= 0, [&](int d) { return __ldg(lp + (size_t)d * HW); }, k, e);
    if (g == 0 && gcls >= 0) atomicAdd(&hist[gcls * D + k], 1u);
    __syncthreads();     // warp 0 reads sm in pixel_class_stats' last merge; the next run overwrites it
  }
  for (int i = threadIdx.x; i < D * D; i += CS_THREADS) {
    const unsigned n = hist[i];
    if (n) atomicAdd(conf + i, (unsigned long long)n);
  }
}

// Pooled (count, sum |E|) tables over the pixels that enter DCA_METRIC_SUM_ABS, binned by the confidence and by the error
// itself.  Both tables live in shared memory (36.9 KB) for the whole grid-stride loop and are flushed with one global
// atomic per non-zero entry, as class_confusion_kernel does.
constexpr int CH_THREADS = 256;
constexpr int CH_ERR_SHIFT = 15;           // 2^-20 px units -> 1/32 px bins
__global__ void __launch_bounds__(CH_THREADS)
confidence_histograms_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const float* __restrict__ peak,
                             unsigned long long* __restrict__ conf_hist, unsigned long long* __restrict__ err_hist,
                             size_t n, float max_valid) {
  __shared__ unsigned long long s_conf[DCA_CONF_BINS][2];
  __shared__ unsigned long long s_err[DCA_ERR_BINS][2];
  for (int i = threadIdx.x; i < 2 * DCA_CONF_BINS; i += CH_THREADS) (&s_conf[0][0])[i] = 0ull;
  for (int i = threadIdx.x; i < 2 * DCA_ERR_BINS; i += CH_THREADS) (&s_err[0][0])[i] = 0ull;
  pdl_wait();
  __syncthreads();
  for (size_t i = (size_t)blockIdx.x * CH_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * CH_THREADS) {
    const float p = __ldg(pred + i), g = __ldg(gt + i);
    if (!gt_valid(g, max_valid) || !isfinite(p)) continue;
    const unsigned long long fix = abs_err_fix(fabsf(__fsub_rn(p, g)));
    const float c = __ldg(peak + i);
    const int cb = (isfinite(c) && c >= 0.f) ? (int)fminf(floorf(__fmul_rn(c, (float)DCA_CONF_BINS)),
                                                          (float)(DCA_CONF_BINS - 1)) : 0;
    const unsigned long long eb64 = fix >> CH_ERR_SHIFT;
    const int eb = eb64 < (unsigned long long)(DCA_ERR_BINS - 1) ? (int)eb64 : DCA_ERR_BINS - 1;
    atomicAdd(&s_conf[cb][0], 1ull);
    atomicAdd(&s_conf[cb][1], fix);
    atomicAdd(&s_err[eb][0], 1ull);
    atomicAdd(&s_err[eb][1], fix);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * DCA_CONF_BINS; i += CH_THREADS) {
    const unsigned long long v = (&s_conf[0][0])[i];
    if (v) atomicAdd(conf_hist + i, v);
  }
  for (int i = threadIdx.x; i < 2 * DCA_ERR_BINS; i += CH_THREADS) {
    const unsigned long long v = (&s_err[0][0])[i];
    if (v) atomicAdd(err_hist + i, v);
  }
}

// Depth errors (DCA_DEPTH_*): the grid and the reduction of disparity_metrics_kernel; the four sums use SUM_ABS's
// fixed-point conversion (fminf(NaN, 2^20) = 2^20)
struct DepthParams {
  float max_valid, fb, doffs, min_depth, max_depth;
};

__global__ void __launch_bounds__(MT_THREADS)
depth_metrics_kernel(const float* __restrict__ pred, const float* __restrict__ gt, unsigned long long* __restrict__ rows,
                     int HW, const DepthParams P) {
  __shared__ unsigned long long red[MT_WARPS][DCA_DEPTH_COUNT];
  pdl_wait();
  const int b = blockIdx.y;
  const float* pb = pred + (size_t)b * HW;
  const float* gb = gt + (size_t)b * HW;
  unsigned long long v[DCA_DEPTH_COUNT];
#pragma unroll
  for (int m = 0; m < DCA_DEPTH_COUNT; ++m) v[m] = 0ull;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += gridDim.x * blockDim.x) {
    const float g = __ldg(gb + i);
    if (!gt_valid(g, P.max_valid)) continue;
    const float zg = __fdiv_rn(P.fb, __fadd_rn(g, P.doffs));
    if (!(zg >= P.min_depth && zg <= P.max_depth)) continue;
    const float pd = __fadd_rn(__ldg(pb + i), P.doffs);
    float zp = (isfinite(pd) && pd > 0.f) ? __fdiv_rn(P.fb, pd) : P.max_depth;
    zp = fminf(fmaxf(zp, P.min_depth), P.max_depth);
    const float e = __fsub_rn(zp, zg);
    const float e2 = __fmul_rn(e, e);
    const float lg = __fsub_rn(logf(zp), logf(zg));
    const float ratio = fmaxf(__fdiv_rn(zp, zg), __fdiv_rn(zg, zp));
    v[DCA_DEPTH_VALID] += 1;
    v[DCA_DEPTH_ABS_REL] += abs_err_fix(__fdiv_rn(fabsf(e), zg));
    v[DCA_DEPTH_SQ_REL] += abs_err_fix(__fdiv_rn(e2, zg));
    v[DCA_DEPTH_SQ] += abs_err_fix(e2);
    v[DCA_DEPTH_LOG_SQ] += abs_err_fix(__fmul_rn(lg, lg));
    v[DCA_DEPTH_A1] += ratio < 1.25f;
    v[DCA_DEPTH_A2] += ratio < 1.5625f;
    v[DCA_DEPTH_A3] += ratio < 1.953125f;
  }
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int m = 0; m < DCA_DEPTH_COUNT; ++m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[m] += __shfl_xor_sync(full, v[m], o);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int m = 0; m < DCA_DEPTH_COUNT; ++m) red[warp][m] = v[m];
  }
  __syncthreads();
  if (threadIdx.x < DCA_DEPTH_COUNT) {
    unsigned long long t = 0;
#pragma unroll
    for (int w = 0; w < MT_WARPS; ++w) t += red[w][threadIdx.x];
    if (t) atomicAdd(rows + (size_t)b * DCA_DEPTH_COUNT + threadIdx.x, t);
  }
}

}  // namespace dca

using namespace dca;

extern "C" int dca_depth_metrics(const float* pred, const float* gt, unsigned long long* rows, int B, int H, int W,
                                 float max_valid, float focal_baseline, float doffs, float min_depth, float max_depth,
                                 void* stream) {
  if (!pred || !gt || !rows || B <= 0 || H <= 0 || W <= 0 || B > 65535 || max_valid != max_valid) return DCA_ERR_ARG;
  if (!(focal_baseline > 0.f) || isinf(focal_baseline) || !isfinite(doffs) || !(min_depth > 0.f) ||
      !(max_depth >= min_depth) || isinf(max_depth))
    return DCA_ERR_ARG;
  if ((long long)H * W > INT_MAX - MT_THREADS) return DCA_ERR_UNSUPPORTED;
  const int HW = H * W;
  int bx = (HW + MT_THREADS - 1) / MT_THREADS;
  const int cap = (4 * dca_num_sms() + B - 1) / B;
  if (bx > cap) bx = cap;
  const DepthParams P = {max_valid, focal_baseline, doffs, min_depth, max_depth};
  dca_launch(depth_metrics_kernel, dim3(bx, B), MT_THREADS, 0, (cudaStream_t)stream, pred, gt, rows, HW, P);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_disparity_metrics(const float* pred, const float* gt, unsigned long long* rows, int B, int H, int W,
                                     float max_valid, void* stream) {
  if (!pred || !gt || !rows || B <= 0 || H <= 0 || W <= 0 || max_valid != max_valid) return DCA_ERR_ARG;
  if (B > 65535 || (long long)H * W > INT_MAX - MT_THREADS) return DCA_ERR_UNSUPPORTED;
  const int HW = H * W;
  const int vec4 = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(gt)) % 16 == 0);
  const int items = vec4 ? HW / 4 : HW;
  int bx = (items + MT_THREADS - 1) / MT_THREADS;
  const int cap = (4 * dca_num_sms() + B - 1) / B;       // about four blocks per SM over the whole batch
  if (bx > cap) bx = cap;
  dca_launch(disparity_metrics_kernel, dim3(bx, B), MT_THREADS, 0, (cudaStream_t)stream, pred, gt, rows, HW, vec4,
             max_valid);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_class_confusion(const float* logits, const float* gt, unsigned long long* conf, int B, int D8, int H8,
                                   int W8, float max_valid, void* stream) {
  if (!logits || !gt || !conf || B <= 0 || D8 <= 0 || H8 <= 0 || W8 <= 0 || max_valid != max_valid) return DCA_ERR_ARG;
  if (D8 > 64 || (long long)H8 * W8 * 64 > INT_MAX || (long long)B * ((H8 * W8 + 31) / 32) > INT_MAX) return DCA_ERR_UNSUPPORTED;
  const int chunks = B * ((H8 * W8 + 31) / 32);
  const int grid = chunks < 8 * dca_num_sms() ? chunks : 8 * dca_num_sms();
  dca_launch(class_confusion_kernel, dim3(grid), CS_THREADS, (size_t)D8 * D8 * sizeof(unsigned), (cudaStream_t)stream,
             logits, gt, conf, B, D8, H8, W8, max_valid);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_confidence_histograms(const float* pred, const float* gt, const float* peak,
                                         unsigned long long* conf_hist, unsigned long long* err_hist, int B, int H,
                                         int W, float max_valid, void* stream) {
  if (!pred || !gt || !peak || !conf_hist || !err_hist || B <= 0 || H <= 0 || W <= 0 || max_valid != max_valid)
    return DCA_ERR_ARG;
  const size_t n = (size_t)B * H * W;
  const size_t want = (n + CH_THREADS - 1) / CH_THREADS;
  const size_t cap = 2 * (size_t)dca_num_sms();          // every block zeroes and flushes 36.9 KB of tables
  dca_launch(confidence_histograms_kernel, dim3((unsigned)(want < cap ? want : cap)), CH_THREADS, 0,
             (cudaStream_t)stream, pred, gt, peak, conf_hist, err_hist, n, max_valid);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
