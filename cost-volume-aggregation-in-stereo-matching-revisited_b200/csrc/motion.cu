// Moving objects between consecutive depth maps: the per-pixel two-frame test and the connected components of the pixels
// that fail it.  Definitions: include/dca_b200.h section (16).
//
//   motion_labels_kernel     one thread per window pixel: back-project, move into the previous camera, project, and
//                            compare the expected disparity with the previous frame's (2r+1)^2 neighbourhood
//   mc_init_kernel           parent = own index for MOVING pixels (-1 otherwise), size = 0, object rows reset
//   mc_merge_kernel          per MOVING pixel, the gated edges to its left and upper neighbours: union by atomicMin of
//                            the roots, so every component's root is its smallest raster index whatever the race order
//   mc_compress_kernel       parent = the root; size[root] += 1
//   mc_tile_kernel           per tile of DCA_MOTION_TILE pixels: the number of kept roots (size >= min_pixels)
//   mc_scan_kernel           one CTA per image: exclusive scan of the tile counts in place, K and dropped
//   mc_number_kernel         per tile: a block scan of the kept roots gives each its id (size[root] <- id, or 0)
//   mc_stats_kernel          per pixel: instance = id of its root; integer atomics into the object rows
//   mc_finalize_kernel       object rows: order-preserving keys back to fp32, rows past K zeroed / NaN
#include <limits.h>
#include <math.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int MO_THREADS = 256;
constexpr int MO_WARPS = MO_THREADS / 32;
constexpr int MO_PER_THREAD = DCA_MOTION_TILE / MO_THREADS;
static_assert(MO_PER_THREAD * MO_THREADS == DCA_MOTION_TILE, "tile = whole passes of the block");
constexpr int MO_SCAN_THREADS = 1024;
constexpr int MO_INTS = 8;
constexpr int MO_EXT = 6;
constexpr float MO_RES_CLAMP = 1048576.f;    // 2^20 px: 2^28 per term, below 2^59 for 2^31 pixels

struct MoCam {
  float fx, fy, cx, cy, u0, v0, fB, doffs;
  float Wf, Hf;
};

struct MoFrames {
  float a[DCA_MOTION_MAX_FRAMES][12];        // T(previous camera <- current camera) per image, row-major
};

__device__ __forceinline__ float mo_row4(const float* m, float a, float b, float c) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
}

__device__ __forceinline__ bool mo_valid(float z) { return isfinite(z) && z > 0.f; }

__device__ __forceinline__ float mo_disp(const MoCam& C, float z) { return __fsub_rn(__fdiv_rn(C.fB, z), C.doffs); }

// order-preserving map of fp32 onto int32 (NaN never reaches it: p is finite for a valid depth)
__device__ __forceinline__ int mo_key(float f) {
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float mo_unkey(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

__global__ void __launch_bounds__(MO_THREADS)
motion_labels_kernel(const float* __restrict__ depth, const float* __restrict__ prev, long long pitch_row,
                     long long pitch_img, int H, int W, const MoCam C, const MoFrames F, float tau, float tau_rel,
                     int radius, unsigned char* __restrict__ label, float* __restrict__ residual) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * MO_THREADS + threadIdx.x;
  const long long HW = (long long)H * W;
  if (e >= HW) return;
  const int y = (int)(e / W), x = (int)(e - (long long)y * W);
  pdl_wait();
  const size_t out = (size_t)b * HW + e;
  const float z = __ldg(depth + (size_t)b * pitch_img + (size_t)y * pitch_row + x);
  unsigned char lab = DCA_MOTION_INVALID;
  float res = __int_as_float(0x7fc00000);
  if (mo_valid(z)) {
    lab = DCA_MOTION_UNSEEN;
    const float* A = F.a[b];
    const float px = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(x), C.u0), C.cx), z), C.fx);
    const float py = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(y), C.v0), C.cy), z), C.fy);
    const float qx = mo_row4(A, px, py, z), qy = mo_row4(A + 4, px, py, z), qz = mo_row4(A + 8, px, py, z);
    if (qz > 0.f) {
      const float mx = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(C.fx, qx), qz), C.cx), C.u0);
      const float my = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(C.fy, qy), qz), C.cy), C.v0);
      const float xf = floorf(__fadd_rn(mx, 0.5f)), yf = floorf(__fadd_rn(my, 0.5f));
      if (xf >= 0.f && xf < C.Wf && yf >= 0.f && yf < C.Hf) {
        const int xm = (int)xf, ym = (int)yf;
        const float ex = mo_disp(C, qz);
        const float tol = fmaxf(tau, __fmul_rn(tau_rel, ex));
        const float* pb = prev + (size_t)b * pitch_img;
        bool any = false, stat = false, appeared = true;
        float best = 0.f;
        for (int dy = -radius; dy <= radius; ++dy) {
          const int yy = ym + dy;
          if (yy < 0 || yy >= H) continue;
          for (int dx = -radius; dx <= radius; ++dx) {
            const int xx = xm + dx;
            if (xx < 0 || xx >= W) continue;
            const float zp = __ldg(pb + (size_t)yy * pitch_row + xx);
            if (!mo_valid(zp)) continue;
            const float s = __fsub_rn(mo_disp(C, zp), ex);
            if (!any || fabsf(s) < fabsf(best)) best = s;
            any = true;
            stat |= fabsf(s) <= tol;
            appeared &= s < -tol;
          }
        }
        if (any) {
          lab = stat ? DCA_MOTION_STATIC : appeared ? DCA_MOTION_APPEARED : DCA_MOTION_BEHIND;
          res = best;
        }
      }
    }
  }
  label[out] = lab;
  residual[out] = res;
}

__device__ __forceinline__ bool mo_moving(unsigned char l) {
  return l == DCA_MOTION_APPEARED || l == DCA_MOTION_BEHIND;
}

__global__ void __launch_bounds__(MO_THREADS)
mc_init_kernel(const unsigned char* __restrict__ label, long long total, int* __restrict__ parent,
               int* __restrict__ size, long long HW, int rows, int* __restrict__ ints, int* __restrict__ ekeys,
               long long* __restrict__ res_sum) {
  const long long e = (long long)blockIdx.x * MO_THREADS + threadIdx.x;
  pdl_wait();
  if (e < total) {
    parent[e] = mo_moving(__ldg(label + e)) ? (int)(e % HW) : -1;
    size[e] = 0;
  }
  if (e < rows) {                                       // object rows: counts 0, mins +max, maxes -max
#pragma unroll
    for (int c = 0; c < MO_INTS; ++c) ints[e * MO_INTS + c] = (c >= 3 && c <= 4) ? INT_MAX : (c >= 5 && c <= 6) ? INT_MIN : 0;
#pragma unroll
    for (int c = 0; c < MO_EXT; ++c) ekeys[e * MO_EXT + c] = (c & 1) ? INT_MIN : INT_MAX;
    res_sum[e] = 0;
  }
}

__device__ __forceinline__ int mc_find(const int* parent, int i) {
  int p = parent[i];
  while (p != i) {
    i = p;
    p = parent[i];
  }
  return i;
}

// hook the larger root under the smaller until both sides share one root
__device__ __forceinline__ void mc_union(int* parent, int a, int b) {
  bool done;
  do {
    a = mc_find(parent, a);
    b = mc_find(parent, b);
    if (a < b) {
      const int old = atomicMin(parent + b, a);
      done = old == b;
      b = old;
    } else if (b < a) {
      const int old = atomicMin(parent + a, b);
      done = old == a;
      a = old;
    } else {
      done = true;
    }
  } while (!done);
}

__global__ void __launch_bounds__(MO_THREADS)
mc_merge_kernel(const float* __restrict__ depth, long long pitch_row, long long pitch_img, int H, int W, const MoCam C,
                float gate, int* __restrict__ parent) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * MO_THREADS + threadIdx.x;
  const long long HW = (long long)H * W;
  if (e >= HW) return;
  const int y = (int)(e / W), x = (int)(e - (long long)y * W);
  pdl_wait();
  int* P = parent + (size_t)b * HW;
  if (P[e] < 0) return;
  const float* db = depth + (size_t)b * pitch_img;
  const float d = mo_disp(C, __ldg(db + (size_t)y * pitch_row + x));
  if (x > 0 && P[e - 1] >= 0 && fabsf(__fsub_rn(d, mo_disp(C, __ldg(db + (size_t)y * pitch_row + x - 1)))) <= gate)
    mc_union(P, (int)e, (int)e - 1);
  if (y > 0 && P[e - W] >= 0 && fabsf(__fsub_rn(d, mo_disp(C, __ldg(db + (size_t)(y - 1) * pitch_row + x)))) <= gate)
    mc_union(P, (int)e, (int)(e - W));
}

__global__ void __launch_bounds__(MO_THREADS)
mc_compress_kernel(long long HW, int* __restrict__ parent, int* __restrict__ size) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * MO_THREADS + threadIdx.x;
  if (e >= HW) return;
  pdl_wait();
  int* P = parent + (size_t)b * HW;
  if (P[e] < 0) return;
  const int r = mc_find(P, (int)e);
  P[e] = r;
  atomicAdd(size + (size_t)b * HW + r, 1);
}

__device__ __forceinline__ bool mc_kept(const int* P, const int* S, long long e, long long HW, int min_pixels) {
  return e < HW && P[e] == (int)e && S[e] >= min_pixels;
}

__global__ void __launch_bounds__(MO_THREADS)
mc_tile_kernel(long long HW, int tiles, const int* __restrict__ parent, const int* __restrict__ size, int min_pixels,
               int* __restrict__ tile) {
  __shared__ int s_warp[MO_WARPS];
  const int b = blockIdx.y, t = threadIdx.x;
  pdl_wait();
  const int* P = parent + (size_t)b * HW;
  const int* S = size + (size_t)b * HW;
  int n = 0;
#pragma unroll
  for (int q = 0; q < MO_PER_THREAD; ++q)
    n += mc_kept(P, S, (long long)blockIdx.x * DCA_MOTION_TILE + q * MO_THREADS + t, HW, min_pixels);
  n = __reduce_add_sync(0xffffffffu, n);
  if ((t & 31) == 0) s_warp[t >> 5] = n;
  __syncthreads();
  if (t == 0) {
    int s = 0;
#pragma unroll
    for (int w = 0; w < MO_WARPS; ++w) s += s_warp[w];
    tile[(size_t)b * tiles + blockIdx.x] = s;
  }
}

// one CTA per image: tile[b][0..tiles) <- exclusive prefix sums; count = min(total, MAX), dropped = the rest
__global__ void __launch_bounds__(MO_SCAN_THREADS)
mc_scan_kernel(int* __restrict__ tile, int tiles, int* __restrict__ count, int* __restrict__ dropped) {
  __shared__ int s_warp[MO_SCAN_THREADS / 32];
  __shared__ int s_carry;
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  int* T = tile + (size_t)b * tiles;
  pdl_wait();
  if (t == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < tiles; base += MO_SCAN_THREADS) {
    const int e = base + t;
    const int x = e < tiles ? T[e] : 0;
    int inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += y;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    int before = s_carry;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (e < tiles) T[e] = before + inc - x;
    __syncthreads();
    if (t == MO_SCAN_THREADS - 1) s_carry = before + inc;
    __syncthreads();
  }
  if (t == 0) {
    const int k = min(s_carry, DCA_MOTION_MAX_OBJECTS);
    count[b] = k;
    dropped[b] = s_carry - k;
  }
}

// per tile: kept roots in raster order get id = 1 + rank (0 past DCA_MOTION_MAX_OBJECTS), stored in size[root]
__global__ void __launch_bounds__(MO_THREADS)
mc_number_kernel(long long HW, int tiles, const int* __restrict__ parent, int* __restrict__ size, int min_pixels,
                 const int* __restrict__ tile) {
  __shared__ int s_cnt[MO_PER_THREAD][MO_WARPS];
  const int b = blockIdx.y, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  pdl_wait();
  const int* P = parent + (size_t)b * HW;
  int* S = size + (size_t)b * HW;
  bool kept[MO_PER_THREAD];
  int incl[MO_PER_THREAD];
#pragma unroll
  for (int q = 0; q < MO_PER_THREAD; ++q) {
    const long long e = (long long)blockIdx.x * DCA_MOTION_TILE + q * MO_THREADS + t;
    kept[q] = mc_kept(P, S, e, HW, min_pixels);
    int c = kept[q];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, c, d);
      if (lane >= d) c += y;
    }
    incl[q] = c;
    if (lane == 31) s_cnt[q][warp] = c;
  }
  __syncthreads();
  int before = tile[(size_t)b * tiles + blockIdx.x];
#pragma unroll
  for (int q = 0; q < MO_PER_THREAD; ++q) {
    int o = before;
#pragma unroll
    for (int w = 0; w < MO_WARPS; ++w) {
      const int c = s_cnt[q][w];
      if (w < warp) o += c;
      before += c;
    }
    const long long e = (long long)blockIdx.x * DCA_MOTION_TILE + q * MO_THREADS + t;
    if (e < HW && P[e] == (int)e) {                   // every root: its id, 0 when not kept
      const int rank = o + incl[q] - 1;
      S[e] = kept[q] && rank < DCA_MOTION_MAX_OBJECTS ? rank + 1 : 0;
    }
  }
}

__global__ void __launch_bounds__(MO_THREADS)
mc_stats_kernel(const float* __restrict__ depth, long long pitch_row, long long pitch_img, const unsigned char* __restrict__ label,
                const float* __restrict__ residual, int H, int W, const MoCam C, const int* __restrict__ parent,
                const int* __restrict__ size, int* __restrict__ instance, int* __restrict__ ints,
                int* __restrict__ ekeys, long long* __restrict__ res_sum) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * MO_THREADS + threadIdx.x;
  const long long HW = (long long)H * W;
  if (e >= HW) return;
  const int y = (int)(e / W), x = (int)(e - (long long)y * W);
  pdl_wait();
  const size_t g = (size_t)b * HW + e;
  const int r = parent[g];
  const int id = r >= 0 ? size[(size_t)b * HW + r] : 0;
  instance[g] = id;
  if (!id) return;
  const size_t row = (size_t)b * DCA_MOTION_MAX_OBJECTS + (id - 1);
  int* I = ints + row * MO_INTS;
  const unsigned char l = label[g];
  atomicAdd(I, 1);
  atomicAdd(I + (l == DCA_MOTION_APPEARED ? 1 : 2), 1);
  atomicMin(I + 3, x);
  atomicMin(I + 4, y);
  atomicMax(I + 5, x);
  atomicMax(I + 6, y);
  const float z = __ldg(depth + (size_t)b * pitch_img + (size_t)y * pitch_row + x);
  const float px = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(x), C.u0), C.cx), z), C.fx);
  const float py = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(y), C.v0), C.cy), z), C.fy);
  int* K = ekeys + row * MO_EXT;
  atomicMin(K + 0, mo_key(px));
  atomicMax(K + 1, mo_key(px));
  atomicMin(K + 2, mo_key(py));
  atomicMax(K + 3, mo_key(py));
  atomicMin(K + 4, mo_key(z));
  atomicMax(K + 5, mo_key(z));
  const float rr = fminf(fmaxf(residual[g], -MO_RES_CLAMP), MO_RES_CLAMP);
  atomicAdd((unsigned long long*)(res_sum + row), (unsigned long long)__float2ll_rn(__fmul_rn(rr, 256.f)));
}

// in place: extent keys (int32) -> fp32; rows past K: ints 0, extent NaN, res_sum 0
__global__ void __launch_bounds__(MO_THREADS)
mc_finalize_kernel(int rows, const int* __restrict__ count, int* __restrict__ ints, int* __restrict__ ekeys,
                   long long* __restrict__ res_sum) {
  const int e = blockIdx.x * MO_THREADS + threadIdx.x;
  if (e >= rows) return;
  pdl_wait();
  const bool live = (e % DCA_MOTION_MAX_OBJECTS) < count[e / DCA_MOTION_MAX_OBJECTS];
#pragma unroll
  for (int c = 0; c < MO_EXT; ++c)
    ekeys[e * MO_EXT + c] = live ? __float_as_int(mo_unkey(ekeys[e * MO_EXT + c])) : 0x7fc00000;
  if (!live) {
#pragma unroll
    for (int c = 0; c < MO_INTS; ++c) ints[e * MO_INTS + c] = 0;
    res_sum[e] = 0;
  }
}

static bool mo_cam_ok(float fx, float fy, float cx, float cy, float fB, float doffs) {
  return isfinite(fx) && fx != 0.f && isfinite(fy) && fy != 0.f && isfinite(cx) && isfinite(cy) && isfinite(doffs) &&
         isfinite(fB) && fB > 0.f;
}

static bool mo_unsupported(int H, int W, int u0, int v0) {
  return H >= (1 << 24) || W >= (1 << 24) || (long long)H * W >= (1ll << 31) || u0 <= -(1 << 24) ||
         u0 >= (1 << 24) || v0 <= -(1 << 24) || v0 >= (1 << 24);
}

static MoCam mo_cam(float fx, float fy, float cx, float cy, int u0, int v0, float fB, float doffs, int H, int W) {
  MoCam C;
  C.fx = fx; C.fy = fy; C.cx = cx; C.cy = cy; C.u0 = (float)u0; C.v0 = (float)v0; C.fB = fB; C.doffs = doffs;
  C.Wf = (float)W; C.Hf = (float)H;
  return C;
}

}  // namespace dca

using namespace dca;

extern "C" int dca_motion_labels(const float* depth, const float* prev, long long pitch_row, long long pitch_img,
                                 int B, int H, int W, float fx, float fy, float cx, float cy, int u0, int v0, float fB,
                                 float doffs, const float* A_host, float tau, float tau_rel, int radius,
                                 unsigned char* label, float* residual, void* stream) {
  if (!depth || !prev || !A_host || !label || !residual) return DCA_ERR_ARG;
  if (B < 1 || B > DCA_MOTION_MAX_FRAMES || H <= 0 || W <= 0 || pitch_row < W || pitch_img < (long long)H * pitch_row)
    return DCA_ERR_ARG;
  if (!mo_cam_ok(fx, fy, cx, cy, fB, doffs) || !(isfinite(tau) && tau >= 0.f) ||
      !(isfinite(tau_rel) && tau_rel >= 0.f) || radius < 0 || radius > DCA_MOTION_MAX_RADIUS)
    return DCA_ERR_ARG;
  for (int i = 0; i < 12 * B; ++i)
    if (!isfinite(A_host[i])) return DCA_ERR_ARG;
  if (mo_unsupported(H, W, u0, v0)) return DCA_ERR_UNSUPPORTED;
  MoFrames F;
  for (int b = 0; b < B; ++b)
    for (int e = 0; e < 12; ++e) F.a[b][e] = A_host[b * 12 + e];
  const MoCam C = mo_cam(fx, fy, cx, cy, u0, v0, fB, doffs, H, W);
  const long long HW = (long long)H * W;
  dca_launch(motion_labels_kernel, dim3((unsigned)((HW + MO_THREADS - 1) / MO_THREADS), B), MO_THREADS, 0,
             (cudaStream_t)stream, depth, prev, pitch_row, pitch_img, H, W, C, F, tau, tau_rel, radius, label,
             residual);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_motion_components(const float* depth, long long pitch_row, long long pitch_img,
                                     const unsigned char* label, const float* residual, int B, int H, int W, float fx,
                                     float fy, float cx, float cy, int u0, int v0, float fB, float doffs, float gate,
                                     int min_pixels, int* instance, int* count, int* dropped, int* ints,
                                     float* extent, long long* res_sum, void* workspace, void* stream) {
  if (!depth || !label || !residual || !instance || !count || !dropped || !ints || !extent || !res_sum || !workspace)
    return DCA_ERR_ARG;
  if (B <= 0 || B > 65535 || H <= 0 || W <= 0 || pitch_row < W || pitch_img < (long long)H * pitch_row)
    return DCA_ERR_ARG;
  if (!mo_cam_ok(fx, fy, cx, cy, fB, doffs) || !(isfinite(gate) && gate >= 0.f) || min_pixels < 1) return DCA_ERR_ARG;
  if (mo_unsupported(H, W, u0, v0)) return DCA_ERR_UNSUPPORTED;
  const MoCam C = mo_cam(fx, fy, cx, cy, u0, v0, fB, doffs, H, W);
  const long long HW = (long long)H * W, total = HW * B;
  const int tiles = (int)((HW + DCA_MOTION_TILE - 1) / DCA_MOTION_TILE);
  const int rows = B * DCA_MOTION_MAX_OBJECTS;
  int* parent = (int*)workspace;
  int* size = parent + total;
  int* tile = size + total;
  int* ekeys = (int*)extent;                          // the keys live in the extent rows until mc_finalize_kernel
  const cudaStream_t st = (cudaStream_t)stream;
  const unsigned px = (unsigned)((HW + MO_THREADS - 1) / MO_THREADS);
  const long long init_n = total > rows ? total : rows;
  dca_launch(mc_init_kernel, dim3((unsigned)((init_n + MO_THREADS - 1) / MO_THREADS)), MO_THREADS, 0, st, label, total,
             parent, size, HW, rows, ints, ekeys, res_sum);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_merge_kernel, dim3(px, B), MO_THREADS, 0, st, depth, pitch_row, pitch_img, H, W, C, gate, parent);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_compress_kernel, dim3(px, B), MO_THREADS, 0, st, HW, parent, size);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_tile_kernel, dim3(tiles, B), MO_THREADS, 0, st, HW, tiles, (const int*)parent, (const int*)size,
             min_pixels, tile);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_scan_kernel, dim3(B), MO_SCAN_THREADS, 0, st, tile, tiles, count, dropped);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_number_kernel, dim3(tiles, B), MO_THREADS, 0, st, HW, tiles, (const int*)parent, size, min_pixels,
             (const int*)tile);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_stats_kernel, dim3(px, B), MO_THREADS, 0, st, depth, pitch_row, pitch_img, label, residual, H, W, C,
             (const int*)parent, (const int*)size, instance, ints, ekeys, res_sum);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(mc_finalize_kernel, dim3((rows + MO_THREADS - 1) / MO_THREADS), MO_THREADS, 0, st, rows,
             (const int*)count, ints, ekeys, res_sum);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
