// Reprojection of a disparity window to metric depth and an ordered 3-D point list.  Definitions: include/dca_b200.h
// section (9).
//
// Two launches, neither waiting on another CTA.  Grid (tiles, B), one CTA per tile of DCA_REPROJECT_TILE window pixels in
// row-major order; the CTA's thread t handles pixels k * RP_THREADS + t, k = 0..RP_PER_THREAD-1, so every load is
// coalesced and the pixel order inside a tile is (k, warp, lane).
//   reproject_count_kernel    keep flags, the tile's kept count into workspace[b][tile], and the depth map
//   reproject_scatter_kernel  the sum of workspace[b][0..tile) (this CTA's first output row), the keep flags again (the
//                             arithmetic is deterministic, so they are the same flags), a block scan of them from warp
//                             ballots, and the scatter of xyz / index; the image's last tile writes count[b]
#include <limits.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int RP_THREADS = 256;
constexpr int RP_WARPS = RP_THREADS / 32;
constexpr int RP_PER_THREAD = DCA_REPROJECT_TILE / RP_THREADS;
static_assert(RP_PER_THREAD * RP_THREADS == DCA_REPROJECT_TILE, "tile = whole passes of the block");

struct ReprojectParams {
  float q[16];          // Q row-major
  float t[12];          // T row-major (has_t)
  int has_t;
  float min_peak, min_depth, max_depth;
};

// one row of a 4-column matrix applied to (a, b, c, 1): ((m0 a + m1 b) + m2 c) + m3, no contraction
__device__ __forceinline__ float row4(const float* m, float a, float b, float c) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
}

struct RpPixel {
  float X, Y, Z;
  bool keep;
};

__device__ __forceinline__ RpPixel rp_pixel(const ReprojectParams& P, const float* __restrict__ disp,
                                            const float* __restrict__ peak, const unsigned char* __restrict__ label,
                                            size_t off, int x, int y, int u0, int v0) {
  const float d = __ldg(disp + off);
  const float u = __int2float_rn(x + u0), v = __int2float_rn(y + v0);
  const float w = row4(P.q + 12, u, v, d);
  RpPixel r;
  r.X = __fdiv_rn(row4(P.q, u, v, d), w);
  r.Y = __fdiv_rn(row4(P.q + 4, u, v, d), w);
  r.Z = __fdiv_rn(row4(P.q + 8, u, v, d), w);
  r.keep = isfinite(d) && w > 0.f && r.Z >= P.min_depth && r.Z <= P.max_depth &&
           (peak == nullptr || __ldg(peak + off) >= P.min_peak) &&
           (label == nullptr || __ldg(label + off) == DCA_LR_CONSISTENT);
  return r;
}

__global__ void __launch_bounds__(RP_THREADS)
reproject_count_kernel(const float* __restrict__ disp, const float* __restrict__ peak,
                       const unsigned char* __restrict__ label, long long pitch_row, long long pitch_img, int H, int W,
                       int u0, int v0, const ReprojectParams P, float* __restrict__ depth, int* __restrict__ workspace,
                       int tiles) {
  __shared__ int s_warp[RP_WARPS];
  const int b = blockIdx.y, t = threadIdx.x;
  const int HW = H * W;
  pdl_wait();
  int n = 0;
#pragma unroll
  for (int k = 0; k < RP_PER_THREAD; ++k) {
    const unsigned p = blockIdx.x * DCA_REPROJECT_TILE + k * RP_THREADS + t;     // < 2^31 + TILE
    if (p < (unsigned)HW) {
      const int y = (int)p / W, x = (int)p - y * W;
      const RpPixel r = rp_pixel(P, disp, peak, label, (size_t)b * pitch_img + (size_t)y * pitch_row + x, x, y, u0, v0);
      n += r.keep;
      if (depth) depth[(size_t)b * HW + p] = r.keep ? r.Z : 0.f;
    }
  }
  n = __reduce_add_sync(0xffffffffu, n);
  if ((t & 31) == 0) s_warp[t >> 5] = n;
  __syncthreads();
  if (t == 0) {
    int s = 0;
#pragma unroll
    for (int w = 0; w < RP_WARPS; ++w) s += s_warp[w];
    workspace[(size_t)b * tiles + blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(RP_THREADS)
reproject_scatter_kernel(const float* __restrict__ disp, const float* __restrict__ peak,
                         const unsigned char* __restrict__ label, long long pitch_row, long long pitch_img, int H, int W,
                         int u0, int v0, const ReprojectParams P, float* __restrict__ xyz, int* __restrict__ index,
                         long long* __restrict__ count, const int* __restrict__ workspace, int tiles) {
  __shared__ int s_base[RP_WARPS];
  __shared__ int s_cnt[RP_PER_THREAD][RP_WARPS];
  const int b = blockIdx.y, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int HW = H * W;
  const unsigned full = 0xffffffffu;
  pdl_wait();

  // first output row of this tile: the kept pixels of the image's earlier tiles
  int base = 0;
  for (int i = t; i < (int)blockIdx.x; i += RP_THREADS) base += workspace[(size_t)b * tiles + i];
  base = __reduce_add_sync(full, base);
  if (lane == 0) s_base[warp] = base;

  RpPixel r[RP_PER_THREAD];
  unsigned ballot[RP_PER_THREAD];
#pragma unroll
  for (int k = 0; k < RP_PER_THREAD; ++k) {
    const unsigned p = blockIdx.x * DCA_REPROJECT_TILE + k * RP_THREADS + t;     // < 2^31 + TILE
    r[k].keep = false;
    if (p < (unsigned)HW) {
      const int y = (int)p / W, x = (int)p - y * W;
      r[k] = rp_pixel(P, disp, peak, label, (size_t)b * pitch_img + (size_t)y * pitch_row + x, x, y, u0, v0);
    }
    ballot[k] = __ballot_sync(full, r[k].keep);
    if (lane == 0) s_cnt[k][warp] = __popc(ballot[k]);
  }
  __syncthreads();
  base = 0;
#pragma unroll
  for (int w = 0; w < RP_WARPS; ++w) base += s_base[w];
  int before = base;                      // kept pixels of the image ahead of pass k's warp 0
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int k = 0; k < RP_PER_THREAD; ++k) {
    int mine = before;
#pragma unroll
    for (int w = 0; w < RP_WARPS; ++w) {
      const int c = s_cnt[k][w];
      if (w < warp) mine += c;
      before += c;
    }
    if (r[k].keep) {
      const int o = mine + __popc(ballot[k] & lt);
      const unsigned p = blockIdx.x * DCA_REPROJECT_TILE + k * RP_THREADS + t;
      float* q = xyz + ((size_t)b * HW + o) * 3;
      if (P.has_t) {
        q[0] = row4(P.t, r[k].X, r[k].Y, r[k].Z);
        q[1] = row4(P.t + 4, r[k].X, r[k].Y, r[k].Z);
        q[2] = row4(P.t + 8, r[k].X, r[k].Y, r[k].Z);
      } else {
        q[0] = r[k].X;
        q[1] = r[k].Y;
        q[2] = r[k].Z;
      }
      index[(size_t)b * HW + o] = (int)p;
    }
  }
  if (blockIdx.x == (unsigned)tiles - 1 && t == 0) count[b] = before;
}

}  // namespace dca

using namespace dca;

extern "C" int dca_reproject(const float* disp, const float* peak, const unsigned char* label, long long pitch_row,
                             long long pitch_img, int B, int H, int W, int u0, int v0, const float* Q_host,
                             const float* T_host, float min_peak, float min_depth, float max_depth, float* depth,
                             float* xyz, int* index, long long* count, int* workspace, void* stream) {
  if (!disp || !Q_host || !xyz || !index || !count || !workspace || B <= 0 || H <= 0 || W <= 0 || B > 65535)
    return DCA_ERR_ARG;
  if ((long long)H * W > INT_MAX || pitch_row < W || pitch_img < (long long)H * pitch_row) return DCA_ERR_ARG;
  if (min_peak != min_peak || min_depth != min_depth || max_depth != max_depth || min_depth > max_depth)
    return DCA_ERR_ARG;
  ReprojectParams P;
  for (int i = 0; i < 16; ++i) P.q[i] = Q_host[i];
  P.has_t = T_host != nullptr;
  for (int i = 0; i < 12; ++i) P.t[i] = T_host ? T_host[i] : 0.f;
  P.min_peak = min_peak;
  P.min_depth = min_depth;
  P.max_depth = max_depth;
  const int tiles = (int)(((long long)H * W + DCA_REPROJECT_TILE - 1) / DCA_REPROJECT_TILE);
  const cudaStream_t st = (cudaStream_t)stream;
  dca_launch(reproject_count_kernel, dim3(tiles, B), RP_THREADS, 0, st, disp, peak, label, pitch_row, pitch_img, H, W,
             u0, v0, P, depth, workspace, tiles);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(reproject_scatter_kernel, dim3(tiles, B), RP_THREADS, 0, st, disp, peak, label, pitch_row, pitch_img, H,
             W, u0, v0, P, xyz, index, count, workspace, tiles);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
