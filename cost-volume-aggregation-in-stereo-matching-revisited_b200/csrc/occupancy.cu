// 2-D occupancy grid: obstacle hits and polar free space of posed depth maps, accumulated in log-odds.
// Definitions: include/dca_b200.h section (17).
//
//   occ_pixels_kernel    one thread per window pixel (blockIdx.y = frame): back-project into the grid frame, classify by
//                        height above the road, and add the quantised weight to the cell's hit count (obstacles) and to
//                        the column's range histogram (obstacles), and the column's near / far range bins (every
//                        counted pixel); integer atomics only
//   occ_columns_kernel   one warp per (frame, column): the first range bin whose obstacle weight reaches the threshold
//   occ_cells_kernel     one thread per cell of the box, x fastest: the frames in order with the cell's state in
//                        registers; a cell no frame updates is neither read nor written
#include <math.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int OC_THREADS = 256;

struct OccGrid {
  int nx, ny, i0, j0, bi, bj;
  float ox, oy, cs;
};

struct OccCam {
  float fx, fy, cx, cy, u0, v0;       // u0, v0 as fp32 (exact: |u0|, |v0| < 2^24)
  float Wf, Hf;                       // window size as fp32 (exact)
  float range_res, max_depth;
  int W, col_width, ncols, nbins;
};

struct OccPixelFrames {
  float m[DCA_OCC_MAX_FRAMES][12];    // grid <- camera per frame, row-major
  float road[DCA_OCC_MAX_FRAMES];     // r_b = M_b[11] - camera_height
  float h_lo, h_hi;
};

struct OccCellFrames {
  float minv[DCA_OCC_MAX_FRAMES][12];   // camera <- grid per frame, row-major
  float road[DCA_OCC_MAX_FRAMES];
  int thr, B;
  float l_hit, l_miss, l_min, l_max;
};

// workspace views: hits [B][bj][bi], occ [B][ncols][nbins], near / far / first [B][ncols].  near holds nbins - k and
// far holds k + 1 under atomicMax, so the zeroed workspace means "no pixel" for both.
struct OccWs {
  int *hits, *occ, *near, *far, *first;
};

__device__ __forceinline__ float oc_row4(const float* m, float a, float b, float c) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
}

__global__ void __launch_bounds__(OC_THREADS)
occ_pixels_kernel(const float* __restrict__ depth, const float* __restrict__ weight, long long pitch_row,
                  long long pitch_img, int H, const OccGrid G, const OccCam C, const OccPixelFrames F, OccWs ws) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * OC_THREADS + threadIdx.x;
  if (e >= (long long)H * C.W) return;
  const int y = (int)(e / C.W), x = (int)(e - (long long)y * C.W);
  const size_t off = (size_t)b * pitch_img + (size_t)y * pitch_row + x;
  const float z = __ldg(depth + off);
  if (!(isfinite(z) && z > 0.f && z <= C.max_depth)) return;
  float w = 1.f;
  if (weight) {
    const float wm = __ldg(weight + off);
    w = wm != wm ? 0.f : fminf(fmaxf(wm, 0.f), 1.f);
  }
  if (!(w > 0.f)) return;
  const float px = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(x), C.u0), C.cx), z), C.fx);
  const float py = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(y), C.v0), C.cy), z), C.fy);
  const float* m = F.m[b];
  const float h = __fsub_rn(oc_row4(m + 8, px, py, z), F.road[b]);
  if (!(h <= F.h_hi)) return;
  const int q = __float2int_rn(__fmul_rn(256.f, w));
  const int c = x / C.col_width;
  const int k = (int)floorf(__fdiv_rn(z, C.range_res));          // z <= max_depth: k < nbins
  const size_t col = (size_t)b * C.ncols + c;
  if (h >= F.h_lo) {
    const float gx = oc_row4(m, px, py, z), gy = oc_row4(m + 4, px, py, z);
    const float fi = floorf(__fadd_rn(__fdiv_rn(__fsub_rn(gx, G.ox), G.cs), 0.5f));
    const float fj = floorf(__fadd_rn(__fdiv_rn(__fsub_rn(gy, G.oy), G.cs), 0.5f));
    // in float, so a NaN or a far point never reaches the int conversion
    if (fi >= (float)G.i0 && fi < (float)G.i0 + (float)G.bi && fj >= (float)G.j0 && fj < (float)G.j0 + (float)G.bj) {
      const int i = (int)fi - G.i0, j = (int)fj - G.j0;
      atomicAdd(ws.hits + ((size_t)b * G.bj + j) * G.bi + i, q);
    }
    atomicAdd(ws.occ + col * C.nbins + k, q);
  }
  atomicMax(ws.near + col, C.nbins - k);
  atomicMax(ws.far + col, k + 1);
}

__global__ void __launch_bounds__(OC_THREADS)
occ_columns_kernel(long long columns, int nbins, int thr, OccWs ws) {
  const long long col = ((long long)blockIdx.x * OC_THREADS + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (col >= columns) return;                                     // whole warps leave together
  const int* o = ws.occ + col * nbins;
  int first = nbins;
  for (int base = 0; base < nbins; base += 32) {
    const int k = base + lane;
    const unsigned hit = __ballot_sync(0xffffffffu, k < nbins && o[k] >= thr);
    if (hit) {
      first = base + __ffs(hit) - 1;
      break;
    }
  }
  if (lane == 0) ws.first[col] = first;
}

__global__ void __launch_bounds__(OC_THREADS)
occ_cells_kernel(float* __restrict__ log_odds, int* __restrict__ updates, const OccGrid G, const OccCam C,
                 const OccCellFrames F, OccWs ws) {
  const long long e = (long long)blockIdx.x * OC_THREADS + threadIdx.x;
  const long long nbox = (long long)G.bi * G.bj;
  if (e >= nbox) return;
  const unsigned eu = (unsigned)e, r = eu / (unsigned)G.bi;       // nbox < 2^31: 32-bit divisions
  const int i = G.i0 + (int)(eu - r * (unsigned)G.bi), j = G.j0 + (int)r;
  const size_t v = (size_t)j * G.nx + i;
  const float sx = __fadd_rn(G.ox, __fmul_rn(G.cs, __int2float_rn(i)));
  const float sy = __fadd_rn(G.oy, __fmul_rn(G.cs, __int2float_rn(j)));
  bool loaded = false;
  float L = 0.f;
  int n = 0;
  for (int b = 0; b < F.B; ++b) {
    bool occupied = __ldg(ws.hits + (size_t)b * nbox + e) >= F.thr, free_ = false;
    if (!occupied) {
      const float* m = F.minv[b];
      const float sz = F.road[b];
      const float Zc = oc_row4(m + 8, sx, sy, sz);
      if (!(Zc > 0.f)) continue;
      const float Xc = oc_row4(m, sx, sy, sz), Yc = oc_row4(m + 4, sx, sy, sz);
      const float x = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(C.fx, Xc), Zc), C.cx), C.u0);
      const float y = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(C.fy, Yc), Zc), C.cy), C.v0);
      const float xf = floorf(__fadd_rn(x, 0.5f)), yf = floorf(__fadd_rn(y, 0.5f));
      if (!(xf >= 0.f && xf < C.Wf && yf >= 0.f && yf < C.Hf)) continue;
      const float kf = floorf(__fdiv_rn(Zc, C.range_res));
      if (!(kf < (float)C.nbins)) continue;
      const int k = (int)kf;
      const size_t col = (size_t)b * C.ncols + (int)xf / C.col_width;
      const int far1 = __ldg(ws.far + col);                      // 0: no counted pixel in the column
      if (far1 == 0) continue;
      const int near = C.nbins - __ldg(ws.near + col), far = far1 - 1;
      free_ = near <= k && k < __ldg(ws.first + col) && k <= far;
    }
    if (!occupied && !free_) continue;
    if (!loaded) {
      loaded = true;
      L = log_odds[v];
      n = updates[v];
    }
    L = occupied ? fminf(__fadd_rn(L, F.l_hit), F.l_max) : fmaxf(__fadd_rn(L, F.l_miss), F.l_min);
    ++n;
  }
  if (loaded) {
    log_odds[v] = L;
    updates[v] = n;
  }
}

static bool oc_finite12(const float* m, int B) {
  for (int e = 0; e < 12 * B; ++e)
    if (!isfinite(m[e])) return false;
  return true;
}

}  // namespace dca

using namespace dca;

extern "C" int dca_occupancy_integrate(float* log_odds, int* updates, int nx, int ny, float ox, float oy,
                                       float cell_size, int i0, int j0, int bi, int bj, const float* depth,
                                       const float* weight, long long pitch_row, long long pitch_img, int B, int H,
                                       int W, float fx, float fy, float cx, float cy, int u0, int v0,
                                       const float* M_host, const float* Minv_host, float camera_height, float h_lo,
                                       float h_hi, int col_width, float range_res, float max_depth, int min_hits,
                                       float l_hit, float l_miss, float l_min, float l_max, void* workspace,
                                       void* stream) {
  if (!log_odds || !updates || !depth || !M_host || !Minv_host || !workspace) return DCA_ERR_ARG;
  if (nx <= 0 || ny <= 0 || H <= 0 || W <= 0 || B < 1 || B > DCA_OCC_MAX_FRAMES || pitch_row < W ||
      pitch_img < (long long)H * pitch_row)
    return DCA_ERR_ARG;
  if (i0 < 0 || j0 < 0 || bi <= 0 || bj <= 0 || (long long)i0 + bi > nx || (long long)j0 + bj > ny) return DCA_ERR_ARG;
  if (ox != ox || oy != oy || camera_height != camera_height || h_lo != h_lo || h_hi != h_hi || !(h_lo < h_hi))
    return DCA_ERR_ARG;
  if (!isfinite(fx) || fx == 0.f || !isfinite(fy) || fy == 0.f || !isfinite(cx) || !isfinite(cy)) return DCA_ERR_ARG;
  if (!oc_finite12(M_host, B) || !oc_finite12(Minv_host, B)) return DCA_ERR_ARG;
  if (!(cell_size > 0.f && isfinite(cell_size)) || !(range_res > 0.f && isfinite(range_res)) ||
      !(max_depth > 0.f && isfinite(max_depth)))
    return DCA_ERR_ARG;
  if (col_width < 1 || col_width > DCA_OCC_MAX_COL_WIDTH || min_hits < 1 || min_hits > DCA_OCC_MAX_HITS)
    return DCA_ERR_ARG;
  if (!(l_hit > 0.f) || !(l_miss < 0.f) || !(l_min < 0.f && l_max > 0.f)) return DCA_ERR_ARG;
  const float nbins_f = floorf(max_depth / range_res) + 1.f;      // host fp32 division: correctly rounded
  if ((long long)nx * ny >= (1ll << 31) || nx >= (1 << 24) || ny >= (1 << 24) || !(nbins_f <= (float)DCA_OCC_MAX_BINS) ||
      (long long)H * W >= DCA_OCC_MAX_PIXELS || H >= (1 << 24) || W >= (1 << 24) || u0 <= -(1 << 24) ||
      u0 >= (1 << 24) || v0 <= -(1 << 24) || v0 >= (1 << 24))
    return DCA_ERR_UNSUPPORTED;
  const int nbins = (int)nbins_f;
  const int ncols = (W + col_width - 1) / col_width;

  const OccGrid G = {nx, ny, i0, j0, bi, bj, ox, oy, cell_size};
  OccCam C;
  C.fx = fx; C.fy = fy; C.cx = cx; C.cy = cy;
  C.u0 = (float)u0; C.v0 = (float)v0; C.Wf = (float)W; C.Hf = (float)H;
  C.range_res = range_res; C.max_depth = max_depth;
  C.W = W; C.col_width = col_width; C.ncols = ncols; C.nbins = nbins;
  OccPixelFrames P;
  OccCellFrames Q;
  for (int b = 0; b < B; ++b) {
    for (int e = 0; e < 12; ++e) {
      P.m[b][e] = M_host[b * 12 + e];
      Q.minv[b][e] = Minv_host[b * 12 + e];
    }
    P.road[b] = Q.road[b] = M_host[b * 12 + 11] - camera_height;      // fp32 subtraction on the host
  }
  for (int b = B; b < DCA_OCC_MAX_FRAMES; ++b) {
    for (int e = 0; e < 12; ++e) P.m[b][e] = Q.minv[b][e] = 0.f;
    P.road[b] = Q.road[b] = 0.f;
  }
  P.h_lo = h_lo; P.h_hi = h_hi;
  Q.thr = 256 * min_hits; Q.B = B;
  Q.l_hit = l_hit; Q.l_miss = l_miss; Q.l_min = l_min; Q.l_max = l_max;

  const long long nbox = (long long)bi * bj;
  OccWs ws;
  ws.hits = (int*)workspace;
  ws.occ = ws.hits + (size_t)B * nbox;
  ws.near = ws.occ + (size_t)B * ncols * nbins;
  ws.far = ws.near + (size_t)B * ncols;
  ws.first = ws.far + (size_t)B * ncols;
  const cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(workspace, 0, DCA_OCC_WORKSPACE_BYTES(B, bi, bj, ncols, nbins), st) != cudaSuccess)
    return DCA_ERR_LAUNCH;
  const dim3 pix((unsigned)(((long long)H * W + OC_THREADS - 1) / OC_THREADS), B);
  occ_pixels_kernel<<<pix, OC_THREADS, 0, st>>>(depth, weight, pitch_row, pitch_img, H, G, C, P, ws);
  DCA_RETURN_IF_LAUNCH_FAILED();
  const long long columns = (long long)B * ncols;
  occ_columns_kernel<<<(unsigned)((columns * 32 + OC_THREADS - 1) / OC_THREADS), OC_THREADS, 0, st>>>(columns, nbins,
                                                                                                    Q.thr, ws);
  DCA_RETURN_IF_LAUNCH_FAILED();
  occ_cells_kernel<<<(unsigned)((nbox + OC_THREADS - 1) / OC_THREADS), OC_THREADS, 0, st>>>(log_odds, updates, G, C, Q,
                                                                                          ws);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
