// The Stixel World from the disparity.  Definitions: include/dca_b200.h section (15).
//
//   dca_ground_profile   V-disparity histogram (int32 atomics), Hough search over (slope, horizon) with one CTA per
//                        (image, horizon row) and a thread per slope, a one-CTA argmax per image, an int64 least-squares
//                        fit of the winning band, and a one-CTA fp64 solve per image.  Integer sums commute, so nothing
//                        depends on the order of the atomics.
//   dca_stixels          column reduction (lower median of each row of a column), the object lut (one CTA per
//                        (image, column), a warp per level, a warp scan along the rows so the writes are coalesced),
//                        and the DP with ONE WARP PER COLUMN: each lane takes every 32nd bottom row n_b of the segment
//                        ending at n_t and a shuffle argmin picks (cost, n_b, c') per class.  The column's prefix sums,
//                        C, the back-pointers and the last-segment disparities stay in shared memory; the warp needs
//                        only __syncwarp between rows.
//   dca_stixel_render    one thread per pixel.
#include <math.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int SX_THREADS = 256;
constexpr int SX_INF = 0x7fffffff;

struct StixelPriors {
  int s_ground, s_object, s_sky, tau, p_seg, p_gravity, p_order, eps_gravity, eps_order;
};

__device__ __forceinline__ bool sx_valid(const float* disp, const float* peak, const unsigned char* label, size_t off,
                                         float min_peak, int max_disp, float& d) {
  d = __ldg(disp + off);
  if (!(d >= 0.f && d < (float)max_disp)) return false;                   // NaN and +-inf fail
  if (peak && !(__ldg(peak + off) >= min_peak)) return false;
  if (label && __ldg(label + off) != DCA_LR_CONSISTENT) return false;
  return true;
}

// E(r, s) = floor(min(r^2, (tau s)^2) 1024 / s^2).  Below the truncation r^2 1024 < 2^44 and s^2 <= 2^28 are exact in
// fp64 and the quotient is below 2^16, so its rounding error (<= 2^-37) is smaller than the distance 1/s^2 >= 2^-28 of a
// non-integer quotient to the next integer: floor of the correctly rounded quotient is the integer floor.
__device__ __forceinline__ int sx_cost(int r, int s, int tau) {
  const int ar = abs(r);
  if (ar >= tau * s) return tau * tau * 1024;
  const long long rr = (long long)ar * ar;
  return (int)floor(__ddiv_rn((double)(rr << 10), (double)((long long)s * s)));
}

// ---- ground profile ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SX_THREADS)
gp_hist_kernel(const float* __restrict__ disp, const float* __restrict__ peak, const unsigned char* __restrict__ label,
               long long pitch_row, long long pitch_img, int H, int W, float min_peak, int max_disp,
               int* __restrict__ hist) {
  const int b = blockIdx.y;
  const long long p = (long long)blockIdx.x * SX_THREADS + threadIdx.x;
  if (p >= (long long)H * W) return;
  const int y = (int)(p / W), x = (int)(p % W);
  float d;
  if (!sx_valid(disp, peak, label, (size_t)b * pitch_img + (size_t)y * pitch_row + x, min_peak, max_disp, d)) return;
  atomicAdd(hist + ((size_t)b * H + y) * max_disp + (int)d, 1);
}

__device__ __forceinline__ float gp_slope(int i) {
  return __fadd_rn(DCA_GROUND_A_MIN, __fmul_rn((float)i, DCA_GROUND_A_STEP));
}

// grid (H, B): CTA j scores every slope for horizon row j
__global__ void __launch_bounds__(SX_THREADS)
gp_hough_kernel(const int* __restrict__ hist, int H, int max_disp, int* __restrict__ scores) {
  const int j = blockIdx.x, b = blockIdx.y, i = threadIdx.x;
  if (i >= DCA_GROUND_NA) return;
  const float a = gp_slope(i);
  const int* hb = hist + (size_t)b * H * max_disp;
  int s = 0;
  for (int y = j + 1; y < H; ++y) {
    const int r = __float2int_rn(__fmul_rn(a, (float)(y - j)));
    if (r - 1 >= max_disp) break;                                         // r grows with y
    const int* row = hb + (size_t)y * max_disp;
#pragma unroll
    for (int dl = -1; dl <= 1; ++dl) {
      const int k = r + dl;
      if (k >= 0 && k < max_disp) s += __ldg(row + k);
    }
  }
  scores[((size_t)b * H + j) * DCA_GROUND_NA + i] = s;
}

// one CTA per image: the largest score, ties to the smallest (i, j)
__global__ void __launch_bounds__(SX_THREADS) gp_select_kernel(const int* __restrict__ scores, int H, int* __restrict__ best) {
  const int b = blockIdx.x;
  const int* sb = scores + (size_t)b * H * DCA_GROUND_NA;
  // key: score high, then (NA - 1 - i) high, then (H - 1 - j) high  ->  one unsigned 64-bit maximum
  unsigned long long key = 0;
  for (int e = threadIdx.x; e < H * DCA_GROUND_NA; e += SX_THREADS) {
    const int j = e / DCA_GROUND_NA, i = e % DCA_GROUND_NA;
    const unsigned long long k = ((unsigned long long)(unsigned)sb[e] << 32) |
                                 ((unsigned long long)(DCA_GROUND_NA - 1 - i) << 16) | (unsigned)(H - 1 - j);
    if (k > key) key = k;
  }
  for (int o = 16; o; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, key, o);
    if (v > key) key = v;
  }
  __shared__ unsigned long long red[SX_THREADS / 32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = key;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < SX_THREADS / 32; ++w)
      if (red[w] > key) key = red[w];
    best[2 * b] = DCA_GROUND_NA - 1 - (int)((key >> 16) & 0xffff);
    best[2 * b + 1] = H - 1 - (int)(key & 0xffff);
  }
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// the inliers of the winning band -> int64 sums n, Sy, Syy, Sq, Syq (one atomic per CTA and sum)
__global__ void __launch_bounds__(SX_THREADS)
gp_fit_kernel(const float* __restrict__ disp, const float* __restrict__ peak, const unsigned char* __restrict__ label,
              long long pitch_row, long long pitch_img, int H, int W, float min_peak, int max_disp,
              const int* __restrict__ best, unsigned long long* __restrict__ sums) {
  const int b = blockIdx.y;
  const long long p = (long long)blockIdx.x * SX_THREADS + threadIdx.x;
  long long v[5] = {0, 0, 0, 0, 0};
  if (p < (long long)H * W) {
    const int y = (int)(p / W), x = (int)(p % W);
    const int i = best[2 * b], j = best[2 * b + 1];
    float d;
    if (y > j && sx_valid(disp, peak, label, (size_t)b * pitch_img + (size_t)y * pitch_row + x, min_peak, max_disp, d)) {
      const int r = __float2int_rn(__fmul_rn(gp_slope(i), (float)(y - j)));
      const int dl = (int)d - r;
      if (dl >= -1 && dl <= 1) {
        const long long q = __float2int_rn(__fmul_rn(d, 256.f));
        v[0] = 1; v[1] = y; v[2] = (long long)y * y; v[3] = q; v[4] = q * y;
      }
    }
  }
  __shared__ long long red[5][SX_THREADS / 32];
#pragma unroll
  for (int t = 0; t < 5; ++t) {
    v[t] = warp_sum_ll(v[t]);
    if ((threadIdx.x & 31) == 0) red[t][threadIdx.x >> 5] = v[t];
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    long long s = 0;
    for (int w = 0; w < SX_THREADS / 32; ++w) s += red[threadIdx.x][w];
    if (s) atomicAdd(sums + 5 * b + threadIdx.x, (unsigned long long)s);
  }
}

// one CTA per image: the fp64 solve, then the profile
__global__ void __launch_bounds__(SX_THREADS)
gp_solve_kernel(const unsigned long long* __restrict__ sums, int H, int min_inliers, float* __restrict__ profile,
                double* __restrict__ line, int* __restrict__ inliers, unsigned char* __restrict__ ok) {
  const int b = blockIdx.x;
  __shared__ double sl[2];
  __shared__ int sok;
  if (threadIdx.x == 0) {
    const unsigned long long* s = sums + 5 * b;
    const double N = __ll2double_rn((long long)s[0]), Y = __ll2double_rn((long long)s[1]);
    const double YY = __ll2double_rn((long long)s[2]), Q = __ll2double_rn((long long)s[3]);
    const double YQ = __ll2double_rn((long long)s[4]);
    const double den = __dsub_rn(__dmul_rn(N, YY), __dmul_rn(Y, Y));
    const double alpha = __ddiv_rn(__dsub_rn(__dmul_rn(N, YQ), __dmul_rn(Y, Q)), den);
    const double beta = __ddiv_rn(__dsub_rn(Q, __dmul_rn(alpha, Y)), N);
    const double a = __dmul_rn(alpha, 1.0 / 256.0), yh = __ddiv_rn(-beta, alpha);
    const int good = (long long)s[0] >= min_inliers && den > 0.0 && a >= DCA_GROUND_MIN_SLOPE && isfinite(yh);
    sok = good;
    sl[0] = good ? a : 0.0;
    sl[1] = good ? yh : 0.0;
    line[2 * b] = sl[0];
    line[2 * b + 1] = sl[1];
    inliers[b] = (int)s[0];
    ok[b] = (unsigned char)good;
  }
  __syncthreads();
  const double a = sl[0], yh = sl[1];
  for (int y = threadIdx.x; y < H; y += SX_THREADS) {
    const double t = __dsub_rn((double)y, yh);
    profile[(size_t)b * H + y] = (sok && t > 0.0) ? __double2float_rn(__dmul_rn(a, t)) : 0.f;
  }
}

// ---- stixels -----------------------------------------------------------------------------------------------
// thread per (image, row, column): the lower median of the row's valid q -> samples[b][k][n], -1 = invalid
__global__ void __launch_bounds__(SX_THREADS)
sx_reduce_kernel(const float* __restrict__ disp, const float* __restrict__ peak, const unsigned char* __restrict__ label,
                 long long pitch_row, long long pitch_img, int H, int W, float min_peak, int width, int max_disp,
                 int ncols, int* __restrict__ samples) {
  const int b = blockIdx.y;
  const long long t = (long long)blockIdx.x * SX_THREADS + threadIdx.x;
  if (t >= (long long)H * ncols) return;
  const int y = (int)(t / ncols), k = (int)(t % ncols);
  const int x0 = k * width, x1 = min(x0 + width, W);
  int v[DCA_STIXEL_MAX_WIDTH];
  int m = 0;
  for (int x = x0; x < x1; ++x) {
    float d;
    if (!sx_valid(disp, peak, label, (size_t)b * pitch_img + (size_t)y * pitch_row + x, min_peak, max_disp, d)) continue;
    const int q = __float2int_rn(__fmul_rn(d, 256.f));
    int e = m++;
    for (; e > 0 && v[e - 1] > q; --e) v[e] = v[e - 1];                     // insertion sort
    v[e] = q;
  }
  int med = -1;
  for (int e = 0; e < DCA_STIXEL_MAX_WIDTH; ++e)                            // constant indexing keeps v in registers
    if (m > 0 && e == (m - 1) / 2) med = v[e];
  samples[((size_t)b * ncols + k) * H + (H - 1 - y)] = med;
}

__device__ __forceinline__ int warp_scan_incl(int v) {
  const int lane = threadIdx.x & 31;
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// grid (ncols, B): lut[b][k][lvl][n] = sum over rows n' < n of the object cost at level lvl
__global__ void __launch_bounds__(SX_THREADS)
sx_lut_kernel(const int* __restrict__ samples, int H, int ncols, int max_disp, int s_object, int tau,
              int* __restrict__ lut) {
  extern __shared__ int q[];
  const int k = blockIdx.x, b = blockIdx.y;
  const size_t col = (size_t)b * ncols + k;
  for (int n = threadIdx.x; n < H; n += SX_THREADS) q[n] = samples[col * H + n];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int lvl = warp; lvl <= max_disp; lvl += SX_THREADS / 32) {
    int* out = lut + (col * (max_disp + 1) + lvl) * (H + 1);
    if (lane == 0) out[0] = 0;
    int carry = 0;
    for (int n0 = 0; n0 < H; n0 += 32) {
      const int n = n0 + lane;
      const int qn = n < H ? q[n] : -1;
      const int s = warp_scan_incl(qn >= 0 ? sx_cost(qn - 256 * lvl, s_object, tau) : 0) + carry;
      if (n < H) out[n + 1] = s;
      carry = __shfl_sync(0xffffffffu, s, 31);
    }
  }
}

__device__ __forceinline__ void sx_take(unsigned long long& best, int cost, int key2) {
  const unsigned long long k = ((unsigned long long)(unsigned)cost << 32) | (unsigned)key2;
  if (k < best) best = k;
}

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
  for (int o = 16; o; o >>= 1) {
    const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
    if (u < v) v = u;
  }
  return v;
}

// grid (ncols, B), one warp.  Shared memory, ints: PV, PQ, PG, PS, PZ [H+1] (prefix sums over rows of: valid rows, q,
// ground cost, sky cost, rows without ground), g [H], C [H][3], BP [H][3] (n_b * 4 + c'), DM [H] (m of the object state)
__global__ void __launch_bounds__(32)
sx_dp_kernel(const int* __restrict__ samples, const int* __restrict__ lut, const float* __restrict__ profile, int H,
             int ncols, int max_disp, const StixelPriors P, int* __restrict__ count, short* __restrict__ bottom,
             short* __restrict__ top, unsigned char* __restrict__ cls, float* __restrict__ sdisp,
             int* __restrict__ free_space) {
  extern __shared__ int sm[];
  int *PV = sm, *PQ = PV + (H + 1), *PG = PQ + (H + 1), *PS = PG + (H + 1), *PZ = PS + (H + 1);
  int *G = PZ + (H + 1), *C = G + H, *BP = C + 3 * H, *DM = BP + 3 * H;
  const int k = blockIdx.x, b = blockIdx.y, lane = threadIdx.x;
  const size_t col = (size_t)b * ncols + k;
  const int* lc = lut + col * (size_t)(max_disp + 1) * (H + 1);

  // prefix sums, 32 rows at a time
  int cv = 0, cq = 0, cg = 0, cs = 0, cz = 0;
  if (lane == 0) PV[0] = PQ[0] = PG[0] = PS[0] = PZ[0] = 0;
  for (int n0 = 0; n0 < H; n0 += 32) {
    const int n = n0 + lane;
    int v = 0, qq = 0, eg = 0, es = 0, z = 0;
    if (n < H) {
      const float dg = __ldg(profile + (size_t)b * H + (H - 1 - n));
      const int g = (isfinite(dg) && dg > 0.f) ? __float2int_rn(__fmul_rn(fminf(dg, (float)max_disp), 256.f)) : 0;
      G[n] = g;
      z = g > 0 ? 0 : 1;
      const int qn = samples[col * H + n];
      if (qn >= 0) {
        v = 1; qq = qn;
        eg = sx_cost(qn - g, P.s_ground, P.tau);
        es = sx_cost(qn, P.s_sky, P.tau);
      }
    }
    v = warp_scan_incl(v) + cv; qq = warp_scan_incl(qq) + cq; eg = warp_scan_incl(eg) + cg;
    es = warp_scan_incl(es) + cs; z = warp_scan_incl(z) + cz;
    if (n < H) { PV[n + 1] = v; PQ[n + 1] = qq; PG[n + 1] = eg; PS[n + 1] = es; PZ[n + 1] = z; }
    cv = __shfl_sync(0xffffffffu, v, 31); cq = __shfl_sync(0xffffffffu, qq, 31);
    cg = __shfl_sync(0xffffffffu, eg, 31); cs = __shfl_sync(0xffffffffu, es, 31);
    cz = __shfl_sync(0xffffffffu, z, 31);
  }
  __syncwarp();

  for (int nt = 0; nt < H; ++nt) {
    unsigned long long bg = ~0ull, bo = ~0ull, bs = ~0ull;
    const int vt = PV[nt + 1], qt = PQ[nt + 1], gt = PG[nt + 1], st = PS[nt + 1], zt = PZ[nt + 1];
    for (int nb = lane; nb <= nt; nb += 32) {
      const int c0 = nb ? C[3 * (nb - 1)] : SX_INF, c1 = nb ? C[3 * (nb - 1) + 1] : SX_INF;
      const int key = nb * 4;
      // ground: all rows with g > 0; only an object (or nothing) below
      if (zt == PZ[nb]) {
        const int data = gt - PG[nb] + P.p_seg;
        if (nb == 0) sx_take(bg, data, key);
        else if (c1 != SX_INF) sx_take(bg, c1 + data, key + DCA_STIXEL_OBJECT);
      }
      // object: at least one valid row
      const int cnt = vt - PV[nb];
      if (cnt > 0) {
        const int m = (2 * (qt - PQ[nb]) + cnt) / (2 * cnt);
        const int lvl = min((m + 128) >> 8, max_disp);
        const int* ll = lc + (size_t)lvl * (H + 1);
        const int data = __ldg(ll + nt + 1) - __ldg(ll + nb) + P.p_seg;
        if (nb == 0) {
          sx_take(bo, data, key);
        } else {
          if (c0 != SX_INF)
            sx_take(bo, c0 + data + (abs(m - G[nb]) > P.eps_gravity ? P.p_gravity : 0), key + DCA_STIXEL_GROUND);
          if (c1 != SX_INF)
            sx_take(bo, c1 + data + (m > DM[nb - 1] + P.eps_order ? P.p_order : 0), key + DCA_STIXEL_OBJECT);
        }
      }
      // sky: anything but sky below
      {
        const int data = st - PS[nb] + P.p_seg;
        if (nb == 0) {
          sx_take(bs, data, key);
        } else {
          if (c0 != SX_INF) sx_take(bs, c0 + data, key + DCA_STIXEL_GROUND);
          if (c1 != SX_INF) sx_take(bs, c1 + data, key + DCA_STIXEL_OBJECT);
        }
      }
    }
    bg = warp_min_u64(bg); bo = warp_min_u64(bo); bs = warp_min_u64(bs);
    if (lane == 0) {
      const unsigned long long bb[3] = {bg, bo, bs};
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        C[3 * nt + c] = bb[c] == ~0ull ? SX_INF : (int)(bb[c] >> 32);
        BP[3 * nt + c] = (int)(bb[c] & 0xffffffffu);
      }
      int m = 0;
      if (bo != ~0ull) {
        const int nb = (int)(bo & 0xffffffffu) >> 2, cnt = vt - PV[nb];
        m = (2 * (qt - PQ[nb]) + cnt) / (2 * cnt);
      }
      DM[nt] = m;
    }
    __syncwarp();
  }

  if (lane == 0) {
    int c = 0;
    for (int e = 1; e < 3; ++e)
      if (C[3 * (H - 1) + e] < C[3 * (H - 1) + c]) c = e;
    const int c_top = c;
    int nsg = 0;
    for (int nt = H - 1; nt >= 0;) {                                        // count the segments
      const int key = BP[3 * nt + c], nb = key >> 2;
      ++nsg;
      c = key & 3;
      nt = nb - 1;
    }
    count[col] = nsg;
    const size_t base = col * H;
    int idx = nsg - 1, fs = H;
    c = c_top;
    for (int nt = H - 1; nt >= 0; --idx) {
      const int key = BP[3 * nt + c], nb = key >> 2;
      bottom[base + idx] = (short)(H - 1 - nb);
      top[base + idx] = (short)(H - 1 - nt);
      cls[base + idx] = (unsigned char)c;
      sdisp[base + idx] = c == DCA_STIXEL_OBJECT ? (float)DM[nt] * (1.f / 256.f) : 0.f;
      if (nb == 0 && c == DCA_STIXEL_GROUND) fs = H - 1 - nt;
      c = key & 3;
      nt = nb - 1;
    }
    free_space[col] = fs;
  }
}

__global__ void __launch_bounds__(SX_THREADS)
sx_render_kernel(const int* __restrict__ count, const short* __restrict__ bottom, const short* __restrict__ top,
                 const unsigned char* __restrict__ cls, const float* __restrict__ sdisp, const float* __restrict__ profile,
                 int H, int W, int width, int ncols, float* __restrict__ out_disp, unsigned char* __restrict__ out_cls) {
  const int b = blockIdx.y;
  const long long p = (long long)blockIdx.x * SX_THREADS + threadIdx.x;
  if (p >= (long long)H * W) return;
  const int y = (int)(p / W), x = (int)(p % W);
  const size_t col = (size_t)b * ncols + x / width, base = col * H;
  const int nsg = min(__ldg(count + col), H);
  float d = 0.f;
  unsigned char c = DCA_STIXEL_SKY;
  for (int i = 0; i < nsg; ++i) {
    if (y >= __ldg(top + base + i) && y <= __ldg(bottom + base + i)) {
      c = __ldg(cls + base + i);
      d = c == DCA_STIXEL_GROUND ? __ldg(profile + (size_t)b * H + y) : c == DCA_STIXEL_OBJECT ? __ldg(sdisp + base + i) : 0.f;
      break;
    }
  }
  out_disp[(size_t)b * H * W + p] = d;
  out_cls[(size_t)b * H * W + p] = c;
}

static unsigned sx_blocks(long long n) { return (unsigned)((n + SX_THREADS - 1) / SX_THREADS); }

static bool sx_map_args(const float* disp, int B, int H, int W, long long pitch_row, long long pitch_img, float min_peak) {
  return disp && B > 0 && B <= 65535 && H > 0 && W > 0 && pitch_row >= W && pitch_img >= (long long)H * pitch_row &&
         !isnan(min_peak);
}

}  // namespace dca

using namespace dca;

extern "C" int dca_ground_profile(const float* disp, const float* peak, const unsigned char* label, long long pitch_row,
                                  long long pitch_img, int B, int H, int W, float min_peak, int max_disp,
                                  int min_inliers, float* profile, double* line, int* inliers, unsigned char* ok,
                                  void* workspace, void* stream) {
  if (!sx_map_args(disp, B, H, W, pitch_row, pitch_img, min_peak)) return DCA_ERR_ARG;
  if (!profile || !line || !inliers || !ok || !workspace) return DCA_ERR_ARG;
  if (max_disp < 1 || max_disp > DCA_STIXEL_MAX_DISP || min_inliers < 1) return DCA_ERR_ARG;
  if ((long long)H * W > INT_MAX || H > DCA_GROUND_MAX_ROWS) return DCA_ERR_UNSUPPORTED;
  unsigned long long* sums = static_cast<unsigned long long*>(workspace);           // [B][5]
  int* best = reinterpret_cast<int*>(sums + 5 * (size_t)B);                         // [B][2]
  int* hist = best + 2 * (size_t)B;                                                 // [B][H][max_disp]
  int* scores = hist + (size_t)B * H * max_disp;                                    // [B][H][NA]
  const cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(workspace, 0, 48ull * B + 4ull * B * H * max_disp, st) != cudaSuccess) return DCA_ERR_LAUNCH;
  const dim3 pix(sx_blocks((long long)H * W), B);
  gp_hist_kernel<<<pix, SX_THREADS, 0, st>>>(disp, peak, label, pitch_row, pitch_img, H, W, min_peak, max_disp, hist);
  DCA_RETURN_IF_LAUNCH_FAILED();
  gp_hough_kernel<<<dim3(H, B), SX_THREADS, 0, st>>>(hist, H, max_disp, scores);
  DCA_RETURN_IF_LAUNCH_FAILED();
  gp_select_kernel<<<B, SX_THREADS, 0, st>>>(scores, H, best);
  DCA_RETURN_IF_LAUNCH_FAILED();
  gp_fit_kernel<<<pix, SX_THREADS, 0, st>>>(disp, peak, label, pitch_row, pitch_img, H, W, min_peak, max_disp, best,
                                           sums);
  DCA_RETURN_IF_LAUNCH_FAILED();
  gp_solve_kernel<<<B, SX_THREADS, 0, st>>>(sums, H, min_inliers, profile, line, inliers, ok);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_stixels(const float* disp, const float* peak, const unsigned char* label, long long pitch_row,
                           long long pitch_img, int B, int H, int W, float min_peak, const float* profile, int width,
                           int max_disp, int s_ground, int s_object, int s_sky, int tau, int p_seg, int p_gravity,
                           int p_order, int eps_gravity, int eps_order, int* count, short* bottom, short* top,
                           unsigned char* cls, float* sdisp, int* free_space, void* workspace, void* stream) {
  if (!sx_map_args(disp, B, H, W, pitch_row, pitch_img, min_peak)) return DCA_ERR_ARG;
  if (!profile || !count || !bottom || !top || !cls || !sdisp || !free_space || !workspace) return DCA_ERR_ARG;
  if (width < 1 || width > DCA_STIXEL_MAX_WIDTH || max_disp < 1 || max_disp > DCA_STIXEL_MAX_DISP) return DCA_ERR_ARG;
  const int sig[3] = {s_ground, s_object, s_sky};
  for (int s : sig)
    if (s < 1 || s > DCA_STIXEL_MAX_SIGMA) return DCA_ERR_ARG;
  if (tau < 1 || tau > DCA_STIXEL_MAX_TAU) return DCA_ERR_ARG;
  const int pri[5] = {p_seg, p_gravity, p_order, eps_gravity, eps_order};
  for (int v : pri)
    if (v < 0 || v > DCA_STIXEL_MAX_PRIOR) return DCA_ERR_ARG;
  if (H > DCA_STIXEL_MAX_ROWS || (long long)H * W > INT_MAX) return DCA_ERR_UNSUPPORTED;
  const int ncols = DCA_STIXEL_COLS(W, width);
  int* samples = static_cast<int*>(workspace);                                      // [B][ncols][H]
  int* lut = samples + (size_t)B * ncols * H;                                       // [B][ncols][max_disp+1][H+1]
  const StixelPriors P = {s_ground, s_object, s_sky, tau, p_seg, p_gravity, p_order, eps_gravity, eps_order};
  const cudaStream_t st = (cudaStream_t)stream;
  sx_reduce_kernel<<<dim3(sx_blocks((long long)H * ncols), B), SX_THREADS, 0, st>>>(
      disp, peak, label, pitch_row, pitch_img, H, W, min_peak, width, max_disp, ncols, samples);
  DCA_RETURN_IF_LAUNCH_FAILED();
  sx_lut_kernel<<<dim3(ncols, B), SX_THREADS, H * sizeof(int), st>>>(samples, H, ncols, max_disp, s_object, tau, lut);
  DCA_RETURN_IF_LAUNCH_FAILED();
  const size_t smem = sizeof(int) * (5 * (size_t)(H + 1) + 8 * (size_t)H);
  sx_dp_kernel<<<dim3(ncols, B), 32, smem, st>>>(samples, lut, profile, H, ncols, max_disp, P, count, bottom, top, cls,
                                                 sdisp, free_space);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_stixel_render(const int* count, const short* bottom, const short* top, const unsigned char* cls,
                                 const float* sdisp, const float* profile, int B, int H, int W, int width, int ncols,
                                 float* out_disp, unsigned char* out_cls, void* stream) {
  if (!count || !bottom || !top || !cls || !sdisp || !profile || !out_disp || !out_cls) return DCA_ERR_ARG;
  if (B <= 0 || B > 65535 || H <= 0 || W <= 0 || width < 1 || width > DCA_STIXEL_MAX_WIDTH) return DCA_ERR_ARG;
  if (ncols != DCA_STIXEL_COLS(W, width)) return DCA_ERR_ARG;
  if (H > DCA_STIXEL_MAX_ROWS || (long long)H * W > INT_MAX) return DCA_ERR_UNSUPPORTED;
  sx_render_kernel<<<dim3(sx_blocks((long long)H * W), B), SX_THREADS, 0, (cudaStream_t)stream>>>(
      count, bottom, top, cls, sdisp, profile, H, W, width, ncols, out_disp, out_cls);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
