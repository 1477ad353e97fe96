// Camera tracking against a fused TSDF volume: raycast model maps and projective point-to-plane ICP.
// Definitions: include/dca_b200.h section (13).
//
//   tsdf_raycast_kernel   one thread per window pixel: the march along the pixel's ray, then depth, camera-frame vertex,
//                         normal and colour of the hit
//   icp_reduce_kernel     per tile of DCA_ICP_TILE source pixels on the level's stride grid: the fixed-point sums of one
//                         iteration (21 of J^T W J, 6 of J^T W r, sum w r^2, sum w, count) into the CTA's workspace row
//   icp_solve_kernel      one CTA: the workspace rows summed (int64, so in any order the same), the 6x6 Cholesky solve
//                         in fp64 and the pose update; it writes the pose, the iteration's stats and the ok flag
#include <math.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int RC_THREADS = 256;
constexpr int ICP_THREADS = 256;
constexpr int ICP_WARPS = ICP_THREADS / 32;
constexpr int ICP_PER_THREAD = DCA_ICP_TILE / ICP_THREADS;
static_assert(ICP_PER_THREAD * ICP_THREADS == DCA_ICP_TILE, "tile = whole passes of the block");
constexpr int ICP_SUMS = 30;                 // 21 + 6 + e + w + count
constexpr int ICP_ROW = DCA_ICP_WORKSPACE_ROW;
static_assert(ICP_SUMS <= ICP_ROW, "a workspace row holds every sum");
constexpr int SOLVE_THREADS = 256;

struct TkGrid {
  int nx, ny, nz;
  float ox, oy, oz, vs;
};

struct RcParams {
  float m[12];                               // camera-to-world 3x4, row-major
  float fx, fy, cx, cy, u0, v0;
  float min_depth, max_depth, min_weight, trunc;
};

__device__ __forceinline__ float tk_row4(const float* m, float a, float b, float c) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
}

__device__ __forceinline__ float tk_lerp(float p, float q, float t) { return __fadd_rn(p, __fmul_rn(t, __fsub_rn(q, p))); }

// trilinear value of plane `pl` in the cell with corner (x0, y0, z0) at fractions (a, b, c)
__device__ __forceinline__ float tk_tri(const float* __restrict__ pl, const TkGrid& G, int x0, int y0, int z0, float a,
                                        float b, float c) {
  const long long sy = G.nx, sz = (long long)G.nx * G.ny;
  const float* p = pl + z0 * sz + y0 * sy + x0;
  const float c00 = tk_lerp(__ldg(p), __ldg(p + 1), a);
  const float c10 = tk_lerp(__ldg(p + sy), __ldg(p + sy + 1), a);
  const float c01 = tk_lerp(__ldg(p + sz), __ldg(p + sz + 1), a);
  const float c11 = tk_lerp(__ldg(p + sz + sy), __ldg(p + sz + sy + 1), a);
  return tk_lerp(tk_lerp(c00, c10, b), tk_lerp(c01, c11, b), c);
}

// a march sample at grid coordinates (gx, gy, gz): false (unknown) when a corner is outside the grid or has weight
// < min_weight, else T = the trilinear tsdf
__device__ __forceinline__ bool tk_sample(const float* __restrict__ vol, long long N, const TkGrid& G, float gx, float gy,
                                          float gz, float min_weight, float& T) {
  const float x0 = floorf(gx), y0 = floorf(gy), z0 = floorf(gz);
  if (!(x0 >= 0.f && x0 < (float)(G.nx - 1) && y0 >= 0.f && y0 < (float)(G.ny - 1) && z0 >= 0.f &&
        z0 < (float)(G.nz - 1)))
    return false;
  const int i = (int)x0, j = (int)y0, k = (int)z0;
  const long long sy = G.nx, sz = (long long)G.nx * G.ny;
  const float* w = vol + N + k * sz + j * sy + i;
#pragma unroll
  for (int dz = 0; dz < 2; ++dz)
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx)
        if (!(__ldg(w + dz * sz + dy * sy + dx) >= min_weight)) return false;
  T = tk_tri(vol, G, i, j, k, __fsub_rn(gx, x0), __fsub_rn(gy, y0), __fsub_rn(gz, z0));
  return true;
}

// the clamped trilinear value of plane `pl` at grid coordinates (gx, gy, gz): each coordinate clamped into
// [0, n - 1], the cell corner min(floor, n - 2)
__device__ __forceinline__ float tk_clamped(const float* __restrict__ pl, const TkGrid& G, float gx, float gy, float gz) {
  gx = fminf(fmaxf(gx, 0.f), (float)(G.nx - 1));
  gy = fminf(fmaxf(gy, 0.f), (float)(G.ny - 1));
  gz = fminf(fmaxf(gz, 0.f), (float)(G.nz - 1));
  const float x0 = fminf(floorf(gx), (float)(G.nx - 2)), y0 = fminf(floorf(gy), (float)(G.ny - 2)),
              z0 = fminf(floorf(gz), (float)(G.nz - 2));
  return tk_tri(pl, G, (int)x0, (int)y0, (int)z0, __fsub_rn(gx, x0), __fsub_rn(gy, y0), __fsub_rn(gz, z0));
}

__global__ void __launch_bounds__(RC_THREADS)
tsdf_raycast_kernel(const float* __restrict__ vol, int planes, long long N, const TkGrid G, int H, int W,
                    const RcParams P, float* __restrict__ depth, long long depth_pitch, float* __restrict__ vertex,
                    long long vertex_pitch, float* __restrict__ normal, long long normal_pitch,
                    unsigned char* __restrict__ rgb, long long rgb_pitch) {
  const long long e = (long long)blockIdx.x * RC_THREADS + threadIdx.x;
  if (e >= (long long)H * W) return;
  const int y = (int)(e / W), x = (int)(e - (long long)y * W);
  const float xn = __fdiv_rn(__fsub_rn(__fadd_rn(__int2float_rn(x), P.u0), P.cx), P.fx);
  const float yn = __fdiv_rn(__fsub_rn(__fadd_rn(__int2float_rn(y), P.v0), P.cy), P.fy);
  const float L = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(xn, xn), __fmul_rn(yn, yn)), 1.f));
  const float half = __fmul_rn(0.5f, G.vs);
  pdl_wait();
  float zh = 0.f;
  bool have = false;
  float zp = 0.f, Tp = 0.f;
  for (float z = P.min_depth; z <= P.max_depth;) {
    const float cxw = __fmul_rn(xn, z), cyw = __fmul_rn(yn, z);
    const float gx = __fdiv_rn(__fsub_rn(tk_row4(P.m, cxw, cyw, z), G.ox), G.vs);
    const float gy = __fdiv_rn(__fsub_rn(tk_row4(P.m + 4, cxw, cyw, z), G.oy), G.vs);
    const float gz = __fdiv_rn(__fsub_rn(tk_row4(P.m + 8, cxw, cyw, z), G.oz), G.vs);
    float T, s;
    if (tk_sample(vol, N, G, gx, gy, gz, P.min_weight, T)) {
      if (have && Tp >= 0.f && T < 0.f) {
        zh = __fadd_rn(zp, __fmul_rn(__fsub_rn(z, zp), __fdiv_rn(Tp, __fsub_rn(Tp, T))));
        break;
      }
      if (have && Tp < 0.f && T >= 0.f) break;
      have = true;
      zp = z;
      Tp = T;
      s = fmaxf(half, __fmul_rn(fabsf(T), P.trunc));
    } else {
      have = false;
      s = P.trunc;
    }
    const float zn = __fadd_rn(z, __fdiv_rn(s, L));
    if (!(zn > z)) break;
    z = zn;
  }
  float out_v[3], out_n[3];
  unsigned char out_c[3] = {0, 0, 0};
  bool hit = zh > 0.f;
  if (hit) {
    const float cxw = __fmul_rn(xn, zh), cyw = __fmul_rn(yn, zh);
    const float gx = __fdiv_rn(__fsub_rn(tk_row4(P.m, cxw, cyw, zh), G.ox), G.vs);
    const float gy = __fdiv_rn(__fsub_rn(tk_row4(P.m + 4, cxw, cyw, zh), G.oy), G.vs);
    const float gz = __fdiv_rn(__fsub_rn(tk_row4(P.m + 8, cxw, cyw, zh), G.oz), G.vs);
    const float ax = __fsub_rn(tk_clamped(vol, G, __fadd_rn(gx, 1.f), gy, gz), tk_clamped(vol, G, __fsub_rn(gx, 1.f), gy, gz));
    const float ay = __fsub_rn(tk_clamped(vol, G, gx, __fadd_rn(gy, 1.f), gz), tk_clamped(vol, G, gx, __fsub_rn(gy, 1.f), gz));
    const float az = __fsub_rn(tk_clamped(vol, G, gx, gy, __fadd_rn(gz, 1.f)), tk_clamped(vol, G, gx, gy, __fsub_rn(gz, 1.f)));
    const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
    hit = len > 0.f;
    if (hit) {
      const float wx = __fdiv_rn(ax, len), wy = __fdiv_rn(ay, len), wz = __fdiv_rn(az, len);
#pragma unroll
      for (int c = 0; c < 3; ++c)
        out_n[c] = __fadd_rn(__fadd_rn(__fmul_rn(P.m[c], wx), __fmul_rn(P.m[4 + c], wy)), __fmul_rn(P.m[8 + c], wz));
      out_v[0] = cxw;
      out_v[1] = cyw;
      out_v[2] = zh;
      if (rgb) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int b8 = __float2int_rn(tk_clamped(vol + (2 + c) * N, G, gx, gy, gz));
          out_c[c] = (unsigned char)min(max(b8, 0), 255);
        }
      }
    }
  }
  if (!hit) {
    zh = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) out_v[c] = out_n[c] = __int_as_float(0x7fc00000);
  }
  depth[(size_t)y * depth_pitch + x] = zh;
  float* vo = vertex + (size_t)y * vertex_pitch + 3 * (size_t)x;
  float* no = normal + (size_t)y * normal_pitch + 3 * (size_t)x;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    vo[c] = out_v[c];
    no[c] = out_n[c];
  }
  if (rgb) {
    unsigned char* co = rgb + (size_t)y * rgb_pitch + 3 * (size_t)x;
#pragma unroll
    for (int c = 0; c < 3; ++c) co[c] = out_c[c];
  }
}

// ---- ICP ----------------------------------------------------------------------------------------------------------
struct IcpPose {
  double a[12];                              // the initial guess A0, row-major 3x4
};

struct IcpFrame {
  float fx, fy, cx, cy, u0, v0, Wf, Hf;
  float max_depth, qmax;
};

__global__ void __launch_bounds__(ICP_THREADS)
icp_reduce_kernel(const float* __restrict__ depth, const float* __restrict__ weight, long long pitch, int H, int W,
                  const float* __restrict__ mvert, long long mvert_pitch, const float* __restrict__ mnorm,
                  long long mnorm_pitch, const IcpFrame F, int stride, int Ws, long long ns, float gate2, int first,
                  const IcpPose A0, const double* __restrict__ pose, long long* __restrict__ workspace) {
  __shared__ long long s_sum[ICP_WARPS][ICP_SUMS];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  pdl_wait();                                // the pose of the previous solve; the workspace it has read
  float A[12];
#pragma unroll
  for (int q = 0; q < 12; ++q) A[q] = __double2float_rn(first ? A0.a[q] : pose[q]);
  long long acc[ICP_SUMS];
#pragma unroll
  for (int q = 0; q < ICP_SUMS; ++q) acc[q] = 0;
#pragma unroll 1
  for (int it = 0; it < ICP_PER_THREAD; ++it) {
    const long long e = (long long)blockIdx.x * DCA_ICP_TILE + it * ICP_THREADS + t;
    if (e >= ns) break;
    const int ys = (int)(e / Ws), xs = (int)(e - (long long)ys * Ws);
    const int x = xs * stride, y = ys * stride;
    const size_t off = (size_t)y * pitch + x;
    const float z = __ldg(depth + off);
    if (!(isfinite(z) && z > 0.f && z <= F.max_depth)) continue;
    float w = 1.f;
    if (weight) {
      const float wm = __ldg(weight + off);
      w = wm != wm ? 0.f : fminf(fmaxf(wm, 0.f), 1.f);
    }
    if (!(w > 0.f)) continue;
    const float px = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(x), F.u0), F.cx), z), F.fx);
    const float py = __fdiv_rn(__fmul_rn(__fsub_rn(__fadd_rn(__int2float_rn(y), F.v0), F.cy), z), F.fy);
    const float qx = tk_row4(A, px, py, z), qy = tk_row4(A + 4, px, py, z), qz = tk_row4(A + 8, px, py, z);
    if (!(qz > 0.f && qz <= F.qmax && fabsf(qx) <= F.qmax && fabsf(qy) <= F.qmax)) continue;
    const float mx = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(F.fx, qx), qz), F.cx), F.u0);
    const float my = __fsub_rn(__fadd_rn(__fdiv_rn(__fmul_rn(F.fy, qy), qz), F.cy), F.v0);
    const float xf = floorf(__fadd_rn(mx, 0.5f)), yf = floorf(__fadd_rn(my, 0.5f));
    if (!(xf >= 0.f && xf < F.Wf && yf >= 0.f && yf < F.Hf)) continue;
    const float* mv = mvert + (size_t)yf * mvert_pitch + 3 * (size_t)xf;
    const float* mn = mnorm + (size_t)yf * mnorm_pitch + 3 * (size_t)xf;
    const float nx = __ldg(mn), ny = __ldg(mn + 1), nz = __ldg(mn + 2);
    const float nn = __fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz));
    if (!(nn <= DCA_ICP_MAX_NORMAL2)) continue;
    const float dx = __fsub_rn(qx, __ldg(mv)), dy = __fsub_rn(qy, __ldg(mv + 1)), dz = __fsub_rn(qz, __ldg(mv + 2));
    const float dd = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    if (!(dd <= gate2)) continue;
    const float r = __fadd_rn(__fadd_rn(__fmul_rn(nx, dx), __fmul_rn(ny, dy)), __fmul_rn(nz, dz));
    const float J[6] = {__fsub_rn(__fmul_rn(qy, nz), __fmul_rn(qz, ny)), __fsub_rn(__fmul_rn(qz, nx), __fmul_rn(qx, nz)),
                        __fsub_rn(__fmul_rn(qx, ny), __fmul_rn(qy, nx)), nx, ny, nz};
    int o = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const float wj = __fmul_rn(w, J[i]);
#pragma unroll
      for (int j = i; j < 6; ++j) acc[o++] += __float2ll_rn(__fmul_rn(__fmul_rn(wj, J[j]), DCA_ICP_SCALE_H));
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) acc[21 + i] += __float2ll_rn(__fmul_rn(__fmul_rn(__fmul_rn(w, J[i]), r), DCA_ICP_SCALE_G));
    acc[27] += __float2ll_rn(__fmul_rn(__fmul_rn(__fmul_rn(w, r), r), DCA_ICP_SCALE_E));
    acc[28] += __float2ll_rn(__fmul_rn(w, DCA_ICP_SCALE_W));
    acc[29] += 1;
  }
#pragma unroll
  for (int q = 0; q < ICP_SUMS; ++q) {
    long long v = acc[q];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (lane == 0) s_sum[warp][q] = v;
  }
  __syncthreads();
  if (t < ICP_ROW) {
    long long v = 0;
    if (t < ICP_SUMS)
#pragma unroll
      for (int w = 0; w < ICP_WARPS; ++w) v += s_sum[w][t];
    workspace[(size_t)blockIdx.x * ICP_ROW + t] = v;
  }
}

// one CTA: sums of the workspace rows -> fp64 system -> Cholesky -> pose update
__global__ void __launch_bounds__(SOLVE_THREADS)
icp_solve_kernel(const long long* __restrict__ workspace, int rows, int first, const IcpPose A0,
                 int min_inliers, double pivot_rel, double* __restrict__ pose, double* __restrict__ stats,
                 int* __restrict__ ok) {
  __shared__ long long s_part[SOLVE_THREADS / 32][32];
  __shared__ long long s_tot[32];
  const int t = threadIdx.x, lane = t & 31, grp = t >> 5;
  pdl_wait();
  long long v = 0;
  if (lane < ICP_SUMS)
    for (int r = grp; r < rows; r += SOLVE_THREADS / 32) v += workspace[(size_t)r * ICP_ROW + lane];
  s_part[grp][lane] = v;
  __syncthreads();
  if (t < 32) {
    long long s = 0;
    for (int g = 0; g < SOLVE_THREADS / 32; ++g) s += s_part[g][t];
    s_tot[t] = s;
  }
  __syncthreads();
  if (t != 0) return;
  double A[12];
  for (int q = 0; q < 12; ++q) A[q] = first ? A0.a[q] : pose[q];
  const long long count = s_tot[29];
  double Hm[6][6], g[6];
  int o = 0;
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) {
      Hm[i][j] = Hm[j][i] = __dmul_rn(__ll2double_rn(s_tot[o]), 1.0 / DCA_ICP_SCALE_H);
      ++o;
    }
  for (int i = 0; i < 6; ++i) g[i] = __dmul_rn(__ll2double_rn(s_tot[21 + i]), 1.0 / DCA_ICP_SCALE_G);
  const double E = __dmul_rn(__ll2double_rn(s_tot[27]), 1.0 / DCA_ICP_SCALE_E);
  const double Sw = __dmul_rn(__ll2double_rn(s_tot[28]), 1.0 / DCA_ICP_SCALE_W);
  int flag = count < (long long)min_inliers ? DCA_ICP_FEW_INLIERS : 0;
  if (!flag) {
    double dmax = 0.0;
    for (int i = 0; i < 6; ++i) dmax = fmax(dmax, Hm[i][i]);
    const double thr = __dmul_rn(pivot_rel, dmax);
    double Lm[6][6];
    for (int j = 0; j < 6 && !flag; ++j) {
      double s = Hm[j][j];
      for (int k = 0; k < j; ++k) s = __dadd_rn(s, -__dmul_rn(Lm[j][k], Lm[j][k]));
      if (!(s > thr)) {
        flag = DCA_ICP_DEGENERATE;
        break;
      }
      const double d = __dsqrt_rn(s);
      Lm[j][j] = d;
      for (int i = j + 1; i < 6; ++i) {
        double u = Hm[i][j];
        for (int k = 0; k < j; ++k) u = __dadd_rn(u, -__dmul_rn(Lm[i][k], Lm[j][k]));
        Lm[i][j] = __ddiv_rn(u, d);
      }
    }
    if (!flag) {
      double yv[6], xi[6];
      for (int i = 0; i < 6; ++i) {
        double u = -g[i];
        for (int k = 0; k < i; ++k) u = __dadd_rn(u, -__dmul_rn(Lm[i][k], yv[k]));
        yv[i] = __ddiv_rn(u, Lm[i][i]);
      }
      for (int i = 5; i >= 0; --i) {
        double u = yv[i];
        for (int k = i + 1; k < 6; ++k) u = __dadd_rn(u, -__dmul_rn(Lm[k][i], xi[k]));
        xi[i] = __ddiv_rn(u, Lm[i][i]);
      }
      // R from the normalised quaternion (1, w / 2)
      const double hx = __dmul_rn(xi[0], 0.5), hy = __dmul_rn(xi[1], 0.5), hz = __dmul_rn(xi[2], 0.5);
      const double nq = __dsqrt_rn(__dadd_rn(__dadd_rn(__dadd_rn(1.0, __dmul_rn(hx, hx)), __dmul_rn(hy, hy)),
                                             __dmul_rn(hz, hz)));
      const double qw = __ddiv_rn(1.0, nq), qx = __ddiv_rn(hx, nq), qy = __ddiv_rn(hy, nq), qz = __ddiv_rn(hz, nq);
      const double xx = __dmul_rn(qx, qx), yy = __dmul_rn(qy, qy), zz = __dmul_rn(qz, qz);
      const double xy = __dmul_rn(qx, qy), xz = __dmul_rn(qx, qz), yz = __dmul_rn(qy, qz);
      const double wx = __dmul_rn(qw, qx), wy = __dmul_rn(qw, qy), wz = __dmul_rn(qw, qz);
      const double R[9] = {__dadd_rn(1.0, -__dmul_rn(2.0, __dadd_rn(yy, zz))), __dmul_rn(2.0, __dadd_rn(xy, -wz)),
                           __dmul_rn(2.0, __dadd_rn(xz, wy)),
                           __dmul_rn(2.0, __dadd_rn(xy, wz)), __dadd_rn(1.0, -__dmul_rn(2.0, __dadd_rn(xx, zz))),
                           __dmul_rn(2.0, __dadd_rn(yz, -wx)),
                           __dmul_rn(2.0, __dadd_rn(xz, -wy)), __dmul_rn(2.0, __dadd_rn(yz, wx)),
                           __dadd_rn(1.0, -__dmul_rn(2.0, __dadd_rn(xx, yy)))};
      double An[12];
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 4; ++j) {
          double s = __dadd_rn(__dadd_rn(__dmul_rn(R[3 * i], A[j]), __dmul_rn(R[3 * i + 1], A[4 + j])),
                               __dmul_rn(R[3 * i + 2], A[8 + j]));
          if (j == 3) s = __dadd_rn(s, xi[3 + i]);
          An[4 * i + j] = s;
        }
      for (int q = 0; q < 12; ++q) A[q] = An[q];
    }
  }
  for (int q = 0; q < 12; ++q) pose[q] = A[q];
  stats[0] = (double)count;
  stats[1] = Sw;
  stats[2] = E;
  stats[3] = (double)flag;
  const int good = (first ? 1 : *ok) && flag == 0;
  *ok = good;
}

static bool tk_grid_ok(const float* vol, int planes, int nx, int ny, int nz, float ox, float oy, float oz, float vs) {
  return vol && (planes == 2 || planes == 5) && nx >= 2 && ny >= 2 && nz >= 2 && isfinite(ox) && isfinite(oy) &&
         isfinite(oz) && isfinite(vs) && vs > 0.f;
}

}  // namespace dca

using namespace dca;

extern "C" int dca_tsdf_raycast(const float* volume, int planes, int nx, int ny, int nz, float ox, float oy, float oz,
                                float voxel_size, float trunc, float min_weight, float fx, float fy, float cx, float cy,
                                int u0, int v0, int H, int W, const float* T_host, float min_depth, float max_depth,
                                float* depth, long long depth_pitch, float* vertex, long long vertex_pitch,
                                float* normal, long long normal_pitch, unsigned char* rgb, long long rgb_pitch,
                                void* stream) {
  if (!tk_grid_ok(volume, planes, nx, ny, nz, ox, oy, oz, voxel_size) || !T_host || !depth || !vertex || !normal)
    return DCA_ERR_ARG;
  if (H <= 0 || W <= 0 || depth_pitch < W || vertex_pitch < 3ll * W || normal_pitch < 3ll * W) return DCA_ERR_ARG;
  if (rgb && (planes != 5 || rgb_pitch < 3ll * W)) return DCA_ERR_ARG;
  if (!(isfinite(trunc) && trunc > 0.f) || min_weight != min_weight || !isfinite(fx) || !isfinite(fy) ||
      !isfinite(cx) || !isfinite(cy) || fx == 0.f || fy == 0.f || !(min_depth >= 0.f) || !isfinite(max_depth) ||
      min_depth > max_depth)
    return DCA_ERR_ARG;
  for (int e = 0; e < 12; ++e)
    if (!isfinite(T_host[e])) return DCA_ERR_ARG;
  const long long N = (long long)nx * ny * nz;
  if (N >= (1ll << 31) || (long long)H * W >= (1ll << 31) || H >= (1 << 24) || W >= (1 << 24) ||
      u0 <= -(1 << 24) || u0 >= (1 << 24) || v0 <= -(1 << 24) || v0 >= (1 << 24) || nx >= (1 << 24) ||
      ny >= (1 << 24) || nz >= (1 << 24))
    return DCA_ERR_UNSUPPORTED;
  RcParams P;
  for (int e = 0; e < 12; ++e) P.m[e] = T_host[e];
  P.fx = fx; P.fy = fy; P.cx = cx; P.cy = cy; P.u0 = (float)u0; P.v0 = (float)v0;
  P.min_depth = min_depth; P.max_depth = max_depth; P.min_weight = min_weight; P.trunc = trunc;
  const TkGrid G = {nx, ny, nz, ox, oy, oz, voxel_size};
  const unsigned blocks = (unsigned)(((long long)H * W + RC_THREADS - 1) / RC_THREADS);
  dca_launch(tsdf_raycast_kernel, dim3(blocks), RC_THREADS, 0, (cudaStream_t)stream, volume, planes, N, G, H, W, P,
             depth, depth_pitch, vertex, vertex_pitch, normal, normal_pitch, rgb, rgb_pitch);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_icp_track(const float* depth, const float* weight, long long pitch, int H, int W, float fx,
                             float fy, float cx, float cy, int u0, int v0, float max_depth, const float* model_vertex,
                             long long vertex_pitch, const float* model_normal, long long normal_pitch,
                             const double* A0_host, int num_levels, const int* level_stride, const int* level_iters,
                             const float* level_gate, int min_inliers, void* workspace, double* pose, double* stats,
                             int* ok, void* stream) {
  if (!depth || !model_vertex || !model_normal || !A0_host || !level_stride || !level_iters || !level_gate ||
      !workspace || !pose || !stats || !ok)
    return DCA_ERR_ARG;
  if (H <= 0 || W <= 0 || pitch < W || vertex_pitch < 3ll * W || normal_pitch < 3ll * W) return DCA_ERR_ARG;
  if (!isfinite(fx) || !isfinite(fy) || !isfinite(cx) || !isfinite(cy) || fx == 0.f || fy == 0.f ||
      !(isfinite(max_depth) && max_depth > 0.f) || min_inliers < 1)
    return DCA_ERR_ARG;
  if (num_levels < 1 || num_levels > DCA_ICP_MAX_LEVELS) return DCA_ERR_ARG;
  for (int l = 0; l < num_levels; ++l)
    if (level_stride[l] < 1 || level_iters[l] < 1 || level_iters[l] > DCA_ICP_MAX_ITERS ||
        !(isfinite(level_gate[l]) && level_gate[l] > 0.f))
      return DCA_ERR_ARG;
  IcpPose A0;
  for (int e = 0; e < 12; ++e) {
    if (!isfinite(A0_host[e])) return DCA_ERR_ARG;
    A0.a[e] = A0_host[e];
  }
  if (max_depth > DCA_ICP_MAX_DEPTH || (long long)H * W > DCA_ICP_MAX_PIXELS || u0 <= -(1 << 24) ||
      u0 >= (1 << 24) || v0 <= -(1 << 24) || v0 >= (1 << 24))
    return DCA_ERR_UNSUPPORTED;
  for (int l = 0; l < num_levels; ++l)
    if (level_gate[l] > DCA_ICP_MAX_GATE) return DCA_ERR_UNSUPPORTED;
  IcpFrame F;
  F.fx = fx; F.fy = fy; F.cx = cx; F.cy = cy; F.u0 = (float)u0; F.v0 = (float)v0; F.Wf = (float)W; F.Hf = (float)H;
  F.max_depth = max_depth; F.qmax = 2.f * max_depth;
  const cudaStream_t st = (cudaStream_t)stream;
  long long* ws = (long long*)workspace;
  int done = 0;
  for (int l = 0; l < num_levels; ++l) {
    const int s = level_stride[l];
    const int Hs = (H + s - 1) / s, Ws = (W + s - 1) / s;
    const long long ns = (long long)Hs * Ws;
    const int rows = (int)((ns + DCA_ICP_TILE - 1) / DCA_ICP_TILE);
    const float g = level_gate[l], gate2 = g * g;
    for (int it = 0; it < level_iters[l]; ++it, ++done) {
      const int first = done == 0;
      dca_launch(icp_reduce_kernel, dim3(rows), ICP_THREADS, 0, st, depth, weight, pitch, H, W, model_vertex,
                 vertex_pitch, model_normal, normal_pitch, F, s, Ws, ns, gate2, first, A0, (const double*)pose, ws);
      DCA_RETURN_IF_LAUNCH_FAILED();
      dca_launch(icp_solve_kernel, dim3(1), SOLVE_THREADS, 0, st, (const long long*)ws, rows, first, A0, min_inliers, (double)DCA_ICP_PIVOT_REL, pose, stats + 4 * done, ok);
      DCA_RETURN_IF_LAUNCH_FAILED();
    }
  }
  return DCA_OK;
}
