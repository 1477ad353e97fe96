// TSDF fusion of posed depth maps into a dense voxel volume and the ordered surface crossings of the fused volume.
// Definitions: include/dca_b200.h section (12).
//
//   tsdf_integrate_kernel   one thread per voxel of the box, x fastest, so the state planes are coalesced; the state of a
//                           voxel is loaded on the first frame that updates it, kept in registers across the B frames
//                           and stored once (a voxel no frame updates is neither read nor written)
//   tsdf_count_kernel       per tile of DCA_TSDF_TILE voxels (linear index order): the number of crossings
//   tsdf_scan_kernel        one CTA: exclusive scan of the tile counts in place (each tile's first output row) and the
//                           total; integer sums, so deterministic, and no CTA waits on another
//   tsdf_scatter_kernel     per tile: the crossings again (deterministic arithmetic, the same ones), a block scan of the
//                           per-voxel counts, and the rows o < capacity
#include <limits.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int TS_THREADS = 256;
constexpr int TS_WARPS = TS_THREADS / 32;
constexpr int TS_PER_THREAD = DCA_TSDF_TILE / TS_THREADS;
static_assert(TS_PER_THREAD * TS_THREADS == DCA_TSDF_TILE, "tile = whole passes of the block");
constexpr int TS_SCAN_THREADS = 1024;

struct TsdfGrid {
  int nx, ny, nz;
  float ox, oy, oz, vs;
};

struct TsdfFrames {
  float t[DCA_TSDF_MAX_FRAMES][12];   // world-to-camera 3x4 per frame, row-major
  float fx, fy, cx, cy, u0, v0;        // u0, v0 as fp32 (exact: |u0|, |v0| < 2^24)
  float Wf, Hf;                        // window size as fp32 (exact)
  float trunc, max_weight, max_depth;
  int B;
};

// one row of a 4-column matrix applied to (a, b, c, 1): ((m0 a + m1 b) + m2 c) + m3, no contraction
__device__ __forceinline__ float ts_row4(const float* m, float a, float b, float c) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
}

__global__ void __launch_bounds__(TS_THREADS)
tsdf_integrate_kernel(float* __restrict__ vol, int planes, long long N, const TsdfGrid G, int i0, int j0, int k0, int bi,
                      int bj, long long nbox, const float* __restrict__ depth, const float* __restrict__ weight,
                      long long pitch_row, long long pitch_img, const unsigned char* __restrict__ rgb, int channels,
                      long long rgb_pitch_row, long long rgb_pitch_img, const TsdfFrames F) {
  const long long e = (long long)blockIdx.x * TS_THREADS + threadIdx.x;
  if (e >= nbox) return;
  const unsigned eu = (unsigned)e, r = eu / (unsigned)bi;      // nbox < 2^31: 32-bit divisions
  const int i = i0 + (int)(eu - r * (unsigned)bi), j = j0 + (int)(r % (unsigned)bj), k = k0 + (int)(r / (unsigned)bj);
  const long long v = ((long long)k * G.ny + j) * G.nx + i;
  const float px = __fadd_rn(G.ox, __fmul_rn(G.vs, __int2float_rn(i)));
  const float py = __fadd_rn(G.oy, __fmul_rn(G.vs, __int2float_rn(j)));
  const float pz = __fadd_rn(G.oz, __fmul_rn(G.vs, __int2float_rn(k)));
  pdl_wait();
  bool loaded = false;
  float T = 0.f, Wt = 0.f, C0 = 0.f, C1 = 0.f, C2 = 0.f;
  for (int b = 0; b < F.B; ++b) {
    const float* m = F.t[b];
    const float Zc = ts_row4(m + 8, px, py, pz);
    if (!(Zc > 0.f)) continue;
    const float Xc = ts_row4(m, px, py, pz), Yc = ts_row4(m + 4, px, py, pz);
    const float x = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(F.fx, Xc), Zc), F.cx), F.u0);
    const float y = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(F.fy, Yc), Zc), F.cy), F.v0);
    const float xf = floorf(__fadd_rn(x, 0.5f)), yf = floorf(__fadd_rn(y, 0.5f));
    if (!(xf >= 0.f && xf < F.Wf && yf >= 0.f && yf < F.Hf)) continue;
    const int xi = (int)xf, yi = (int)yf;
    const size_t off = (size_t)b * pitch_img + (size_t)yi * pitch_row + xi;
    const float z = __ldg(depth + off);
    if (!(isfinite(z) && z > 0.f && z <= F.max_depth)) continue;
    float w = 1.f;
    if (weight) {
      const float wm = __ldg(weight + off);
      w = wm != wm ? 0.f : fminf(fmaxf(wm, 0.f), 1.f);
    }
    if (!(w > 0.f)) continue;
    const float sdf = __fsub_rn(z, Zc);
    if (sdf < -F.trunc) continue;
    const float f = fminf(1.f, __fdiv_rn(sdf, F.trunc));
    if (!loaded) {
      loaded = true;
      T = vol[v];
      Wt = vol[N + v];
      if (planes == 5) {
        C0 = vol[2 * N + v];
        C1 = vol[3 * N + v];
        C2 = vol[4 * N + v];
      }
    }
    const float Wn = __fadd_rn(Wt, w);
    T = __fdiv_rn(__fadd_rn(__fmul_rn(T, Wt), __fmul_rn(f, w)), Wn);
    if (planes == 5) {
      const unsigned char* q = rgb + (size_t)b * rgb_pitch_img + (size_t)yi * rgb_pitch_row + (size_t)xi * channels;
      C0 = __fdiv_rn(__fadd_rn(__fmul_rn(C0, Wt), __fmul_rn(__int2float_rn(__ldg(q)), w)), Wn);
      C1 = __fdiv_rn(__fadd_rn(__fmul_rn(C1, Wt), __fmul_rn(__int2float_rn(__ldg(q + 1)), w)), Wn);
      C2 = __fdiv_rn(__fadd_rn(__fmul_rn(C2, Wt), __fmul_rn(__int2float_rn(__ldg(q + 2)), w)), Wn);
    }
    Wt = fminf(Wn, F.max_weight);
  }
  if (loaded) {
    vol[v] = T;
    vol[N + v] = Wt;
    if (planes == 5) {
      vol[2 * N + v] = C0;
      vol[3 * N + v] = C1;
      vol[4 * N + v] = C2;
    }
  }
}

// crossings of voxel v = (i, j, k) along x, y, z as bits 0..2
__device__ __forceinline__ unsigned ts_crossings(const float* __restrict__ vol, long long N, const TsdfGrid& G,
                                                 long long v, int i, int j, int k, float min_weight) {
  const float wv = __ldg(vol + N + v);
  if (!(wv >= min_weight)) return 0u;
  const bool neg = __ldg(vol + v) < 0.f;
  unsigned m = 0u;
  const long long step[3] = {1, G.nx, (long long)G.nx * G.ny};
  const bool inside[3] = {i + 1 < G.nx, j + 1 < G.ny, k + 1 < G.nz};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (!inside[a]) continue;
    const long long n = v + step[a];
    if (__ldg(vol + N + n) >= min_weight && (__ldg(vol + n) < 0.f) != neg) m |= 1u << a;
  }
  return m;
}

__device__ __forceinline__ void ts_coords(const TsdfGrid& G, long long v, int& i, int& j, int& k) {
  const unsigned vu = (unsigned)v, r = vu / (unsigned)G.nx;    // v < N < 2^31: 32-bit divisions
  i = (int)(vu - r * (unsigned)G.nx);
  j = (int)(r % (unsigned)G.ny);
  k = (int)(r / (unsigned)G.ny);
}

__global__ void __launch_bounds__(TS_THREADS)
tsdf_count_kernel(const float* __restrict__ vol, long long N, const TsdfGrid G, float min_weight,
                  long long* __restrict__ workspace) {
  __shared__ int s_warp[TS_WARPS];
  const int t = threadIdx.x;
  pdl_wait();
  int n = 0;
#pragma unroll
  for (int q = 0; q < TS_PER_THREAD; ++q) {
    const long long v = (long long)blockIdx.x * DCA_TSDF_TILE + q * TS_THREADS + t;
    if (v < N) {
      int i, j, k;
      ts_coords(G, v, i, j, k);
      n += __popc(ts_crossings(vol, N, G, v, i, j, k, min_weight));
    }
  }
  n = __reduce_add_sync(0xffffffffu, n);
  if ((t & 31) == 0) s_warp[t >> 5] = n;
  __syncthreads();
  if (t == 0) {
    int s = 0;
#pragma unroll
    for (int w = 0; w < TS_WARPS; ++w) s += s_warp[w];
    workspace[blockIdx.x] = s;
  }
}

// one CTA: workspace[0..tiles) <- exclusive prefix sums, count <- the total
__global__ void __launch_bounds__(TS_SCAN_THREADS)
tsdf_scan_kernel(long long* __restrict__ workspace, int tiles, long long* __restrict__ count) {
  __shared__ long long s_warp[TS_SCAN_THREADS / 32];
  __shared__ long long s_carry;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  pdl_wait();
  if (t == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < tiles; base += TS_SCAN_THREADS) {
    const int e = base + t;
    const long long x = e < tiles ? workspace[e] : 0;
    long long inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const long long y = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += y;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    long long before = s_carry;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (e < tiles) workspace[e] = before + inc - x;
    __syncthreads();                                   // every thread has read s_carry and s_warp
    if (t == TS_SCAN_THREADS - 1) s_carry = before + inc;
    __syncthreads();
  }
  if (t == 0) *count = s_carry;
}

__global__ void __launch_bounds__(TS_THREADS)
tsdf_scatter_kernel(const float* __restrict__ vol, int planes, long long N, const TsdfGrid G, float min_weight,
                    const long long* __restrict__ workspace, long long capacity, float* __restrict__ xyz,
                    float* __restrict__ normal, unsigned char* __restrict__ rgb) {
  __shared__ int s_cnt[TS_PER_THREAD][TS_WARPS];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const unsigned full = 0xffffffffu;
  pdl_wait();
  unsigned mask[TS_PER_THREAD];
  int incl[TS_PER_THREAD];
#pragma unroll
  for (int q = 0; q < TS_PER_THREAD; ++q) {
    const long long v = (long long)blockIdx.x * DCA_TSDF_TILE + q * TS_THREADS + t;
    mask[q] = 0u;
    if (v < N) {
      int i, j, k;
      ts_coords(G, v, i, j, k);
      mask[q] = ts_crossings(vol, N, G, v, i, j, k, min_weight);
    }
    int c = __popc(mask[q]);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(full, c, d);
      if (lane >= d) c += y;
    }
    incl[q] = c;
    if (lane == 31) s_cnt[q][warp] = c;
  }
  __syncthreads();
  long long before = workspace[blockIdx.x];          // crossings of the grid ahead of pass q's warp 0
#pragma unroll
  for (int q = 0; q < TS_PER_THREAD; ++q) {
    long long o = before;
#pragma unroll
    for (int w = 0; w < TS_WARPS; ++w) {
      const int c = s_cnt[q][w];
      if (w < warp) o += c;
      before += c;
    }
    unsigned m = mask[q];
    if (!m) continue;
    o += incl[q] - __popc(m);
    const long long v = (long long)blockIdx.x * DCA_TSDF_TILE + q * TS_THREADS + t;
    int i, j, k;
    ts_coords(G, v, i, j, k);
    const float p[3] = {__fadd_rn(G.ox, __fmul_rn(G.vs, __int2float_rn(i))),
                        __fadd_rn(G.oy, __fmul_rn(G.vs, __int2float_rn(j))),
                        __fadd_rn(G.oz, __fmul_rn(G.vs, __int2float_rn(k)))};
    const float Tv = __ldg(vol + v);
    const long long step[3] = {1, G.nx, (long long)G.nx * G.ny};
    float nrm[3] = {0.f, 0.f, 0.f};
    if (normal) {
      const long long sx = (long long)G.nx * G.ny;
      const float gx = __fsub_rn(__ldg(vol + v + (i + 1 < G.nx ? 1 : 0)), __ldg(vol + v - (i > 0 ? 1 : 0)));
      const float gy = __fsub_rn(__ldg(vol + v + (j + 1 < G.ny ? G.nx : 0)), __ldg(vol + v - (j > 0 ? G.nx : 0)));
      const float gz = __fsub_rn(__ldg(vol + v + (k + 1 < G.nz ? sx : 0)), __ldg(vol + v - (k > 0 ? sx : 0)));
      const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)), __fmul_rn(gz, gz)));
      if (len > 0.f) {
        nrm[0] = __fdiv_rn(gx, len);
        nrm[1] = __fdiv_rn(gy, len);
        nrm[2] = __fdiv_rn(gz, len);
      }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (!(m & (1u << a))) continue;
      if (o < capacity) {
        const long long n = v + step[a];
        const float tt = __fdiv_rn(Tv, __fsub_rn(Tv, __ldg(vol + n)));
        float* dst = xyz + o * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) dst[c] = c == a ? __fadd_rn(p[c], __fmul_rn(tt, G.vs)) : p[c];
        if (normal) {
#pragma unroll
          for (int c = 0; c < 3; ++c) normal[o * 3 + c] = nrm[c];
        }
        if (rgb) {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float cv = __ldg(vol + (2 + c) * N + v), cn = __ldg(vol + (2 + c) * N + n);
            const int b8 = __float2int_rn(__fadd_rn(cv, __fmul_rn(tt, __fsub_rn(cn, cv))));
            rgb[o * 3 + c] = (unsigned char)min(max(b8, 0), 255);
          }
        }
      }
      ++o;
    }
  }
}

static bool ts_grid_ok(const float* vol, int planes, int nx, int ny, int nz, float ox, float oy, float oz, float vs) {
  return vol && (planes == 2 || planes == 5) && nx > 0 && ny > 0 && nz > 0 && ox == ox && oy == oy && oz == oz &&
         vs > 0.f;
}

}  // namespace dca

using namespace dca;

extern "C" int dca_tsdf_integrate(float* volume, int planes, int nx, int ny, int nz, float ox, float oy, float oz,
                                  float voxel_size, int i0, int j0, int k0, int bi, int bj, int bk, const float* depth,
                                  const float* weight, long long pitch_row, long long pitch_img, int B, int H, int W,
                                  const unsigned char* rgb, int channels, long long rgb_pitch_row,
                                  long long rgb_pitch_img, float fx, float fy, float cx, float cy, int u0, int v0,
                                  const float* T_host, float trunc, float max_weight, float max_depth, void* stream) {
  if (!ts_grid_ok(volume, planes, nx, ny, nz, ox, oy, oz, voxel_size) || !depth || !T_host) return DCA_ERR_ARG;
  if (B < 1 || B > DCA_TSDF_MAX_FRAMES || H <= 0 || W <= 0 || pitch_row < W || pitch_img < (long long)H * pitch_row)
    return DCA_ERR_ARG;
  if (i0 < 0 || j0 < 0 || k0 < 0 || bi <= 0 || bj <= 0 || bk <= 0 || (long long)i0 + bi > nx ||
      (long long)j0 + bj > ny || (long long)k0 + bk > nz)
    return DCA_ERR_ARG;
  if ((planes == 5) != (rgb != nullptr)) return DCA_ERR_ARG;
  if (rgb && (channels < 3 || channels > 4 || rgb_pitch_row < (long long)W * channels ||
              rgb_pitch_img < (long long)H * rgb_pitch_row))
    return DCA_ERR_ARG;
  if (fx != fx || fy != fy || cx != cx || cy != cy || !(trunc > 0.f) || !(max_weight > 0.f) || max_depth != max_depth)
    return DCA_ERR_ARG;
  const long long N = (long long)nx * ny * nz;
  if (N >= (1ll << 31) || H >= (1 << 24) || W >= (1 << 24) || u0 <= -(1 << 24) || u0 >= (1 << 24) ||
      v0 <= -(1 << 24) || v0 >= (1 << 24))
    return DCA_ERR_UNSUPPORTED;
  TsdfFrames F;
  for (int b = 0; b < B; ++b)
    for (int e = 0; e < 12; ++e) F.t[b][e] = T_host[b * 12 + e];
  F.fx = fx; F.fy = fy; F.cx = cx; F.cy = cy;
  F.u0 = (float)u0; F.v0 = (float)v0; F.Wf = (float)W; F.Hf = (float)H;
  F.trunc = trunc; F.max_weight = max_weight; F.max_depth = max_depth; F.B = B;
  const TsdfGrid G = {nx, ny, nz, ox, oy, oz, voxel_size};
  const long long nbox = (long long)bi * bj * bk;
  const unsigned blocks = (unsigned)((nbox + TS_THREADS - 1) / TS_THREADS);
  dca_launch(tsdf_integrate_kernel, dim3(blocks), TS_THREADS, 0, (cudaStream_t)stream, volume, planes, N, G, i0, j0, k0,
             bi, bj, nbox, depth, weight, pitch_row, pitch_img, rgb, channels, rgb_pitch_row, rgb_pitch_img, F);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_tsdf_count_surface(const float* volume, int planes, int nx, int ny, int nz, float min_weight,
                                      long long* workspace, long long* count, void* stream) {
  if (!ts_grid_ok(volume, planes, nx, ny, nz, 0.f, 0.f, 0.f, 1.f) || !workspace || !count || min_weight != min_weight)
    return DCA_ERR_ARG;
  const long long N = (long long)nx * ny * nz;
  if (N >= (1ll << 31)) return DCA_ERR_UNSUPPORTED;
  const int tiles = (int)((N + DCA_TSDF_TILE - 1) / DCA_TSDF_TILE);
  const TsdfGrid G = {nx, ny, nz, 0.f, 0.f, 0.f, 1.f};
  const cudaStream_t st = (cudaStream_t)stream;
  dca_launch(tsdf_count_kernel, dim3(tiles), TS_THREADS, 0, st, volume, N, G, min_weight, workspace);
  DCA_RETURN_IF_LAUNCH_FAILED();
  dca_launch(tsdf_scan_kernel, dim3(1), TS_SCAN_THREADS, 0, st, workspace, tiles, count);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_tsdf_extract_surface(const float* volume, int planes, int nx, int ny, int nz, float ox, float oy,
                                        float oz, float voxel_size, float min_weight, const long long* workspace,
                                        long long capacity, float* xyz, float* normal, unsigned char* rgb,
                                        void* stream) {
  if (!ts_grid_ok(volume, planes, nx, ny, nz, ox, oy, oz, voxel_size) || !workspace || min_weight != min_weight ||
      capacity < 0 || (capacity > 0 && !xyz) || (rgb && planes != 5))
    return DCA_ERR_ARG;
  const long long N = (long long)nx * ny * nz;
  if (N >= (1ll << 31)) return DCA_ERR_UNSUPPORTED;
  const int tiles = (int)((N + DCA_TSDF_TILE - 1) / DCA_TSDF_TILE);
  const TsdfGrid G = {nx, ny, nz, ox, oy, oz, voxel_size};
  dca_launch(tsdf_scatter_kernel, dim3(tiles), TS_THREADS, 0, (cudaStream_t)stream, volume, planes, N, G, min_weight,
             workspace, capacity, xyz, normal, rgb);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
