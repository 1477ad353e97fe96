// LiDAR guidance of the cost volume (Guided Stereo Matching, Poggi et al. CVPR 2019).  Definitions: include/dca_b200.h
// section (14).  The modulation itself lives in the guided instantiations of the volume kernels (volume.cu).
//
//   dca_lidar_hints     three launches: fill the z-buffer, scatter every point with a 64-bit atomicMin of
//                       (Z bits << 32 | point index), then turn each pixel's winner into its disparity.  The atomics
//                       commute, so the map does not depend on their order.
//   dca_guide_quarter   one launch: per 1/4-res pixel the largest valid hint of its 4x4 block, divided by 4.
#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int GD_THREADS = 256;
constexpr unsigned long long GD_EMPTY = ~0ull;

struct LidarParams {
  float m[12];                       // velo_to_rect, row-major 3x4
  float fx, fy, cx, cy, fB, doffs, min_depth, max_depth;
  int view, y0, x0, h, w, v_origin, H, W, stride;
};

// one row of the 3x4 transform: fmaf(m2, z, fmaf(m1, y, fmaf(m0, x, m3)))
__device__ __forceinline__ float lidar_row(const float* m, float x, float y, float z) {
  return fmaf(m[2], z, fmaf(m[1], y, fmaf(m[0], x, m[3])));
}

__global__ void __launch_bounds__(GD_THREADS) lidar_fill_kernel(unsigned long long* __restrict__ zbuf, size_t n) {
  for (size_t i = (size_t)blockIdx.x * GD_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * GD_THREADS)
    zbuf[i] = GD_EMPTY;
}

// grid (blocks, B): image b walks its points offsets[b] .. offsets[b+1] (clamped to [0, N])
__global__ void __launch_bounds__(GD_THREADS)
lidar_scatter_kernel(const float* __restrict__ pts, const int* __restrict__ offsets, int N, const LidarParams P,
                     unsigned long long* __restrict__ zbuf) {
  const int b = blockIdx.y;
  const int lo = min(max(__ldg(offsets + b), 0), N), hi = min(max(__ldg(offsets + b + 1), lo), N);
  for (long long p = lo + (long long)blockIdx.x * GD_THREADS + threadIdx.x; p < hi; p += (long long)gridDim.x * GD_THREADS) {
    const float* q = pts + (size_t)p * P.stride;
    const float x = __ldg(q), y = __ldg(q + 1), z = __ldg(q + 2);
    const float X = lidar_row(P.m, x, y, z), Y = lidar_row(P.m + 4, x, y, z), Z = lidar_row(P.m + 8, x, y, z);
    if (!(Z >= P.min_depth && Z <= P.max_depth)) continue;          // also drops NaN
    float u = __fadd_rn(__fdiv_rn(__fmul_rn(P.fx, X), Z), P.cx);
    const float v = __fadd_rn(__fdiv_rn(__fmul_rn(P.fy, Y), Z), P.cy);
    const float disp = __fsub_rn(__fdiv_rn(P.fB, Z), P.doffs);
    if (P.view) u = __fsub_rn(u, disp);
    const float fu = floorf(__fadd_rn(u, 0.5f)), fv = floorf(__fadd_rn(v, 0.5f));
    if (!(fu >= (float)P.x0 && fu < (float)(P.x0 + P.w))) continue;
    if (!(fv >= (float)P.v_origin && fv < (float)(P.v_origin + P.h))) continue;
    const int col = (int)fu, row = P.y0 + ((int)fv - P.v_origin);
    const unsigned long long key = ((unsigned long long)__float_as_uint(Z) << 32) | (unsigned)p;
    atomicMin(zbuf + ((size_t)b * P.H + row) * P.W + col, key);
  }
}

__global__ void __launch_bounds__(GD_THREADS)
lidar_finalise_kernel(const unsigned long long* __restrict__ zbuf, size_t n, float fB, float doffs,
                      float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * GD_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * GD_THREADS) {
    const unsigned long long key = zbuf[i];
    out[i] = key == GD_EMPTY ? 0.f : __fsub_rn(__fdiv_rn(fB, __uint_as_float((unsigned)(key >> 32))), doffs);
  }
}

// one thread per 1/4-res pixel
__global__ void __launch_bounds__(GD_THREADS)
guide_quarter_kernel(const float* __restrict__ hints, int B, int H, int W, float maxdisp, float* __restrict__ hq) {
  const int Hq = H / 4, Wq = W / 4;
  const size_t n = (size_t)B * Hq * Wq;
  for (size_t i = (size_t)blockIdx.x * GD_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * GD_THREADS) {
    const int j = (int)(i % Wq);
    const size_t r = i / Wq;
    const int iq = (int)(r % Hq), b = (int)(r / Hq);
    const float* src = hints + ((size_t)b * H + 4 * iq) * W + 4 * j;
    float m = 0.f;
#pragma unroll
    for (int y = 0; y < 4; ++y)
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        const float v = __ldg(src + (size_t)y * W + x);
        if (v > 0.f && v < maxdisp && v > m) m = v;             // finite and 0 < v < maxdisp; NaN fails v > 0
      }
    hq[i] = m * 0.25f;
  }
}

static int gd_blocks(size_t n) {
  const size_t cap = (size_t)dca_num_sms() * 8, need = (n + GD_THREADS - 1) / GD_THREADS;
  return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

}  // namespace dca

using namespace dca;

static bool gd_small(int v) { return v > -(1 << 24) && v < (1 << 24); }     // exact as fp32

extern "C" int dca_lidar_hints(const float* points, int stride, const int* offsets, int B, int N,
                               const float* velo_to_rect_host, float fx, float fy, float cx, float cy, float fB,
                               float doffs, int view, int y0, int x0, int h, int w, int v_origin, float min_depth,
                               float max_depth, unsigned long long* zbuf, float* out, int H, int W, void* stream) {
  if (!offsets || !velo_to_rect_host || !zbuf || !out || (N > 0 && !points)) return DCA_ERR_ARG;
  if ((stride != 3 && stride != 4) || B <= 0 || N < 0 || H <= 0 || W <= 0 || (view != 0 && view != 1)) return DCA_ERR_ARG;
  if (!(y0 >= 0 && x0 >= 0 && h > 0 && w > 0 && y0 <= H - h && x0 <= W - w)) return DCA_ERR_ARG;
  if (!(isfinite(fx) && fx != 0.f && isfinite(fy) && fy != 0.f && isfinite(cx) && isfinite(cy) && isfinite(fB) &&
        fB > 0.f && isfinite(doffs)))
    return DCA_ERR_ARG;
  if (!(min_depth > 0.f && max_depth >= min_depth && isfinite(max_depth))) return DCA_ERR_ARG;
  LidarParams P;
  for (int i = 0; i < 12; ++i) {
    P.m[i] = velo_to_rect_host[i];
    if (!isfinite(P.m[i])) return DCA_ERR_ARG;
  }
  if (!gd_small(H) || !gd_small(W) || !gd_small(v_origin) || !gd_small(v_origin + h)) return DCA_ERR_UNSUPPORTED;
  P.fx = fx; P.fy = fy; P.cx = cx; P.cy = cy; P.fB = fB; P.doffs = doffs; P.min_depth = min_depth;
  P.max_depth = max_depth; P.view = view; P.y0 = y0; P.x0 = x0; P.h = h; P.w = w; P.v_origin = v_origin; P.H = H;
  P.W = W; P.stride = stride;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)B * H * W;
  lidar_fill_kernel<<<gd_blocks(n), GD_THREADS, 0, st>>>(zbuf, n);
  DCA_RETURN_IF_LAUNCH_FAILED();
  if (N > 0) {
    lidar_scatter_kernel<<<dim3(gd_blocks((size_t)N), B), GD_THREADS, 0, st>>>(points, offsets, N, P, zbuf);
    DCA_RETURN_IF_LAUNCH_FAILED();
  }
  lidar_finalise_kernel<<<gd_blocks(n), GD_THREADS, 0, st>>>(zbuf, n, fB, doffs, out);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_guide_quarter(const float* hints, int B, int H, int W, float maxdisp, float* hq, void* stream) {
  if (!hints || !hq || B <= 0 || H <= 0 || W <= 0 || H % 4 || W % 4 || !(maxdisp > 0.f)) return DCA_ERR_ARG;
  const size_t n = (size_t)B * (H / 4) * (W / 4);
  guide_quarter_kernel<<<gd_blocks(n), GD_THREADS, 0, (cudaStream_t)stream>>>(hints, B, H, W, maxdisp, hq);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
