// Confidence-weighted fast global smoother guided by the left image.  Definition: include/dca_b200.h section (11).
//
//   wls_prepare_kernel  grid (tiles of WP_THREADS pixels, B).  Per pixel: the confidence c, U = c d into `refined`,
//                       V = c into `support`, and the weights to the right and lower neighbours (0 at the last column /
//                       row, so e_{n-1} = 0 needs no special case in the solves).  The weights do not change across
//                       iterations; only lambda_t does.
//   A pass (rows or columns, template ROWS) solves every line partitioned into segments of at most DCA_WLS_SEGMENT
//   elements separated by single separator elements, in up to three launches:
//   wls_seg_kernel      (only with separators) grid (ceil(lines / 32), segments, B), one warp per 32 lines of one
//                       segment, lane = line.  The warp stages the segment's U, V and weights in shared memory with
//                       coalesced loads (a row segment is contiguous; a column segment is 32 adjacent columns per
//                       element), then runs the forward and the reverse elimination sweeps in one loop (two independent
//                       chains) and writes the segment's 8 boundary values.
//   wls_reduce_kernel   (only with separators) one thread per line: the tridiagonal system of the separators, written
//                       into U / V at the separators (or finalised there in the last pass).
//   wls_solve_kernel    as wls_seg_kernel: Thomas elimination of the segment with the separator values folded into its
//                       end rows, p / g_U / g_V kept in the shared tiles, then U and V stored back (the last column pass
//                       writes support = V and refined = U / V or disp).
#include <limits.h>
#include <math.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int WP_THREADS = 256;
constexpr int WK = DCA_WLS_SEGMENT;  // separator spacing: a segment holds at most WK elements
constexpr int TP = WK + 1;           // shared tile pitch: odd, so lane-strided column reads are conflict-free
constexpr int WL = 32;               // lines per warp

__global__ void __launch_bounds__(WP_THREADS)
wls_prepare_kernel(const float* __restrict__ disp, const float* __restrict__ peak, const unsigned char* __restrict__ label,
                   long long pitch_row, long long pitch_img, int H, int W, const unsigned char* __restrict__ guide, int C,
                   long long g_row, long long g_img, const float* __restrict__ lut, float* __restrict__ U,
                   float* __restrict__ V, float* __restrict__ wh, float* __restrict__ wv) {
  const int b = blockIdx.y;
  const int HW = H * W;
  const long long pl = (long long)blockIdx.x * WP_THREADS + threadIdx.x;
  pdl_wait();
  if (pl >= HW) return;
  const int p = (int)pl;
  const int y = p / W, x = p - y * W;
  const long long off = (long long)b * pitch_img + (long long)y * pitch_row + x;
  const float d = disp[off];
  float c = 1.f;
  if (peak) c = fminf(fmaxf(peak[off], 0.f), 1.f);               // fmaxf(NaN, 0) = 0
  if (label && label[off] != DCA_LR_CONSISTENT) c = 0.f;
  if (!isfinite(d) || !(c > 0.f)) c = 0.f;                        // also turns a -0 into +0
  const size_t o = (size_t)b * HW + p;
  U[o] = c > 0.f ? __fmul_rn(c, d) : 0.f;
  V[o] = c;
  const unsigned char* g = guide + (long long)b * g_img + (long long)y * g_row + (long long)x * C;
  float h = 0.f, v = 0.f;
  if (x + 1 < W) {
    int s = 0;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const int q = (int)g[ch] - (int)g[C + ch];
      s += q * q;
    }
    h = __ldg(lut + s);
  }
  if (y + 1 < H) {
    int s = 0;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const int q = (int)g[ch] - (int)g[g_row + ch];
      s += q * q;
    }
    v = __ldg(lut + s);
  }
  wh[o] = h;
  wv[o] = v;
}

// Lines of one pass: element i of line l of image b at b img + l lstride + i estride (rows: lstride W, estride 1;
// columns: lstride 1, estride W).
struct WlsLines {
  int n, nl, S;                 // line length, lines per image, segments per line
  long long img, lstride, estride;
};

__device__ __forceinline__ float wls_rcp(float x) { return __frcp_rn(x); }

// t[l][koff + k] = src[l lstride + (i0 + k) estride], l < nlines, k < len <= WK + 1; src points at line l0 of image b.
// The loads of WB lines (rows) or WB elements (columns) are issued together before any of them is stored, so a tile
// costs a few L2 round trips, not one per element.
constexpr int WB = 16;

template <bool ROWS>
__device__ __forceinline__ void wls_tile_load(float (*t)[TP], const float* __restrict__ src, const WlsLines& L,
                                              int nlines, int i0, int len, int koff) {
  const int lane = threadIdx.x;
  if (ROWS) {
    for (int l0 = 0; l0 < nlines; l0 += WB) {
      float v[WB][3];
#pragma unroll
      for (int j = 0; j < WB; ++j) {
        const float* p = src + (long long)(l0 + j) * L.lstride + i0;
#pragma unroll
        for (int h = 0; h < 3; ++h) v[j][h] = (l0 + j < nlines && lane + 32 * h < len) ? p[lane + 32 * h] : 0.f;
      }
#pragma unroll
      for (int j = 0; j < WB; ++j)
#pragma unroll
        for (int h = 0; h < 3; ++h)
          if (l0 + j < nlines && lane + 32 * h < len) t[l0 + j][koff + lane + 32 * h] = v[j][h];
    }
  } else if (lane < nlines) {
    const float* p = src + lane + (long long)i0 * L.estride;
    for (int k0 = 0; k0 < len; k0 += WB) {
      float v[WB];
#pragma unroll
      for (int j = 0; j < WB; ++j) v[j] = k0 + j < len ? p[(long long)(k0 + j) * L.estride] : 0.f;
#pragma unroll
      for (int j = 0; j < WB; ++j)
        if (k0 + j < len) t[lane][koff + k0 + j] = v[j];
    }
  }
}

template <bool ROWS>
__device__ __forceinline__ void wls_tile_store(const float (*t)[TP], float* __restrict__ dst, const WlsLines& L,
                                               int nlines, int i0, int len) {
  const int lane = threadIdx.x;
  if (ROWS) {
    float* p = dst + i0;
    for (int l = 0; l < nlines; ++l, p += L.lstride)
      for (int k = lane; k < len; k += WL) p[k] = t[l][k];
  } else if (lane < nlines) {
    float* p = dst + lane + (long long)i0 * L.estride;
    for (int k = 0; k < len; ++k, p += L.estride) *p = t[lane][k];
  }
}

// the segment of a block: elements [a, c); weights w[a-1 .. c-1] in tw[0 .. len] (tw[0] = 0 for the first segment)
template <bool ROWS>
__device__ __forceinline__ void wls_load_segment(float (*tu)[TP], float (*tv)[TP], float (*tw)[TP],
                                                 const float* U, const float* V, const float* w, const WlsLines& L,
                                                 size_t base, int nlines, int a, int len) {
  wls_tile_load<ROWS>(tu, U + base, L, nlines, a, len, 0);
  wls_tile_load<ROWS>(tv, V + base, L, nlines, a, len, 0);
  if (a > 0) {
    wls_tile_load<ROWS>(tw, w + base, L, nlines, a - 1, len + 1, 0);
  } else {
    wls_tile_load<ROWS>(tw, w + base, L, nlines, 0, len, 1);
    tw[threadIdx.x][0] = 0.f;
  }
}

template <bool ROWS>
__global__ void __launch_bounds__(WL)
wls_seg_kernel(const float* __restrict__ U, const float* __restrict__ V, const float* __restrict__ w,
               float* __restrict__ R, WlsLines L, float lam) {
  __shared__ float tu[WL][TP], tv[WL][TP], tw[WL][TP];
  const int lane = threadIdx.x, l0 = blockIdx.x * WL, s = blockIdx.y, b = blockIdx.z;
  const int nlines = min(WL, L.nl - l0);
  const int a = s * WK, len = (s + 1 < L.S ? a + WK - 1 : L.n) - a;
  const size_t base = (size_t)b * L.img + (size_t)l0 * L.lstride;
  pdl_wait();
  wls_load_segment<ROWS>(tu, tv, tw, U, V, w, L, base, nlines, a, len);
  __syncwarp();
  if (lane >= nlines) return;
  const float eL = __fmul_rn(lam, tw[lane][0]), eR = __fmul_rn(lam, tw[lane][len]);
  // forward sweep (k) and reverse sweep (j = len-1-k) of the segment's own matrix, interleaved
  float ep = eL, pp = 0.f, gu = 0.f, gv = 0.f, gphi = 0.f, m = 1.f;
  float en = 0.f, rn = 0.f, hu = 0.f, hv = 0.f, hpsi = 0.f, q = 1.f;
  for (int k = 0; k < len; ++k) {
    const float e = __fmul_rn(lam, tw[lane][k + 1]);
    m = wls_rcp(__fsub_rn(__fadd_rn(__fadd_rn(1.f, ep), e), __fmul_rn(ep, pp)));
    gu = __fmul_rn(__fadd_rn(tu[lane][k], __fmul_rn(ep, gu)), m);
    gv = __fmul_rn(__fadd_rn(tv[lane][k], __fmul_rn(ep, gv)), m);
    gphi = k == 0 ? __fmul_rn(eL, m) : __fmul_rn(__fmul_rn(ep, gphi), m);
    pp = __fmul_rn(e, m);
    ep = e;
    const int j = len - 1 - k;
    const float ej = __fmul_rn(lam, tw[lane][j + 1]), ejm = __fmul_rn(lam, tw[lane][j]);
    q = wls_rcp(__fsub_rn(__fadd_rn(__fadd_rn(1.f, ejm), ej), __fmul_rn(ej, rn)));
    hu = __fmul_rn(__fadd_rn(tu[lane][j], __fmul_rn(ej, hu)), q);
    hv = __fmul_rn(__fadd_rn(tv[lane][j], __fmul_rn(ej, hv)), q);
    hpsi = k == 0 ? __fmul_rn(eR, q) : __fmul_rn(__fmul_rn(ej, hpsi), q);
    rn = __fmul_rn(ejm, q);
    en = ej;
  }
  (void)en;
  float* r = R + (((size_t)b * L.nl + l0 + lane) * L.S + s) * 8;
  r[0] = hu;                     // y_U at the first element
  r[1] = hv;                     // y_V at the first element
  r[2] = __fmul_rn(eL, q);       // phi at the first element
  r[3] = hpsi;                   // psi at the first element
  r[4] = gu;                     // y_U at the last element
  r[5] = gv;                     // y_V at the last element
  r[6] = gphi;                   // phi at the last element
  r[7] = __fmul_rn(eR, m);       // psi at the last element
}

template <bool ROWS>
__global__ void __launch_bounds__(WL)
wls_reduce_kernel(float* __restrict__ U, float* __restrict__ V, const float* __restrict__ w, float* __restrict__ R,
                  WlsLines L, float lam, int final_pass, const float* __restrict__ disp, long long pitch_row,
                  long long pitch_img, float min_support) {
  const int line = blockIdx.x * WL + threadIdx.x, b = blockIdx.y;
  pdl_wait();
  if (line >= L.nl) return;
  const size_t base = (size_t)b * L.img + (size_t)line * L.lstride;
  float* Rl = R + ((size_t)b * L.nl + line) * L.S * 8;
  float pp = 0.f, gU = 0.f, gV = 0.f;
  for (int s = 0; s + 1 < L.S; ++s) {
    const int c = (s + 1) * WK - 1;
    float* r = Rl + s * 8;
    const float* rn = r + 8;
    const float em = __fmul_rn(lam, w[base + (size_t)(c - 1) * L.estride]);
    const float ec = __fmul_rn(lam, w[base + (size_t)c * L.estride]);
    const float lo = __fmul_rn(em, r[6]), up = __fmul_rn(ec, rn[3]);
    const float D = __fsub_rn(__fsub_rn(__fadd_rn(__fadd_rn(1.f, em), ec), __fmul_rn(em, r[7])), __fmul_rn(ec, rn[2]));
    const float rU = __fadd_rn(__fadd_rn(U[base + (size_t)c * L.estride], __fmul_rn(em, r[4])), __fmul_rn(ec, rn[0]));
    const float rV = __fadd_rn(__fadd_rn(V[base + (size_t)c * L.estride], __fmul_rn(em, r[5])), __fmul_rn(ec, rn[1]));
    const float m = wls_rcp(__fsub_rn(D, __fmul_rn(lo, pp)));
    pp = __fmul_rn(up, m);
    gU = __fmul_rn(__fadd_rn(rU, __fmul_rn(lo, gU)), m);
    gV = __fmul_rn(__fadd_rn(rV, __fmul_rn(lo, gV)), m);
    r[0] = pp;
    r[1] = gU;
    r[2] = gV;
  }
  float xU = 0.f, xV = 0.f;
  for (int s = L.S - 2; s >= 0; --s) {
    const int c = (s + 1) * WK - 1;
    float* r = Rl + s * 8;
    xU = __fadd_rn(r[1], __fmul_rn(r[0], xU));
    xV = __fadd_rn(r[2], __fmul_rn(r[0], xV));
    r[3] = xU;
    r[4] = xV;
    const size_t i = base + (size_t)c * L.estride;
    V[i] = xV;
    if (!final_pass) {
      U[i] = xU;
    } else {      // the last pass is a column pass: line = x, element = y
      U[i] = xV >= min_support ? __fdiv_rn(xU, xV)
                               : disp[(long long)b * pitch_img + (long long)c * pitch_row + line];
    }
  }
}

template <bool ROWS>
__global__ void __launch_bounds__(WL)
wls_solve_kernel(float* __restrict__ U, float* __restrict__ V, const float* __restrict__ w,
                 const float* __restrict__ R, WlsLines L, float lam, int final_pass, const float* __restrict__ disp,
                 long long pitch_row, long long pitch_img, float min_support) {
  __shared__ float tu[WL][TP], tv[WL][TP], tw[WL][TP];
  const int lane = threadIdx.x, l0 = blockIdx.x * WL, s = blockIdx.y, b = blockIdx.z;
  const int nlines = min(WL, L.nl - l0);
  const int a = s * WK, len = (s + 1 < L.S ? a + WK - 1 : L.n) - a;
  const size_t base = (size_t)b * L.img + (size_t)l0 * L.lstride;
  pdl_wait();
  wls_load_segment<ROWS>(tu, tv, tw, U, V, w, L, base, nlines, a, len);
  __syncwarp();
  if (lane < nlines) {
    const float* r = R + (((size_t)b * L.nl + l0 + lane) * L.S + s) * 8;
    const float eL = __fmul_rn(lam, tw[lane][0]);
    if (s > 0) {                 // the separator to the left, x = r[-8 + 3], r[-8 + 4]
      tu[lane][0] = __fadd_rn(tu[lane][0], __fmul_rn(eL, r[-5]));
      tv[lane][0] = __fadd_rn(tv[lane][0], __fmul_rn(eL, r[-4]));
    }
    if (s + 1 < L.S) {           // the separator to the right
      const float eR = __fmul_rn(lam, tw[lane][len]);
      tu[lane][len - 1] = __fadd_rn(tu[lane][len - 1], __fmul_rn(eR, r[3]));
      tv[lane][len - 1] = __fadd_rn(tv[lane][len - 1], __fmul_rn(eR, r[4]));
    }
    float ep = eL, pp = 0.f, gu = 0.f, gv = 0.f;
    for (int k = 0; k < len; ++k) {
      const float e = __fmul_rn(lam, tw[lane][k + 1]);
      const float m = wls_rcp(__fsub_rn(__fadd_rn(__fadd_rn(1.f, ep), e), __fmul_rn(ep, pp)));
      gu = __fmul_rn(__fadd_rn(tu[lane][k], __fmul_rn(ep, gu)), m);
      gv = __fmul_rn(__fadd_rn(tv[lane][k], __fmul_rn(ep, gv)), m);
      pp = __fmul_rn(e, m);
      ep = e;
      tw[lane][k + 1] = pp;
      tu[lane][k] = gu;
      tv[lane][k] = gv;
    }
    float un = 0.f, vn = 0.f;
    for (int k = len - 1; k >= 0; --k) {
      const float pk = tw[lane][k + 1];
      un = __fadd_rn(tu[lane][k], __fmul_rn(pk, un));
      vn = __fadd_rn(tv[lane][k], __fmul_rn(pk, vn));
      tu[lane][k] = un;
      tv[lane][k] = vn;
    }
  }
  __syncwarp();
  if (!ROWS && final_pass) {     // support = V, refined = U / V or disp; line = x, element = y
    if (lane < nlines) {
      const size_t o = base + lane + (size_t)a * L.estride;
      const float* dp = disp + (long long)b * pitch_img + (long long)a * pitch_row + l0 + lane;
      for (int k = 0; k < len; ++k) {
        const float u = tu[lane][k], v = tv[lane][k];
        V[o + (size_t)k * L.estride] = v;
        U[o + (size_t)k * L.estride] = v >= min_support ? __fdiv_rn(u, v) : dp[(long long)k * pitch_row];
      }
    }
    return;
  }
  wls_tile_store<ROWS>(tu, U + base, L, nlines, a, len);
  wls_tile_store<ROWS>(tv, V + base, L, nlines, a, len);
}

template <bool ROWS>
static int wls_pass(float* U, float* V, const float* w, float* R, const WlsLines& L, float lam, int final_pass,
                    const float* disp, long long pitch_row, long long pitch_img, float min_support, int B,
                    cudaStream_t st) {
  const unsigned groups = (unsigned)((L.nl + WL - 1) / WL);
  if (L.S > 1) {
    dca_launch(wls_seg_kernel<ROWS>, dim3(groups, L.S, B), WL, 0, st, (const float*)U, (const float*)V, w, R, L, lam);
    DCA_RETURN_IF_LAUNCH_FAILED();
    dca_launch(wls_reduce_kernel<ROWS>, dim3(groups, B), WL, 0, st, U, V, w, R, L, lam, final_pass, disp, pitch_row,
               pitch_img, min_support);
    DCA_RETURN_IF_LAUNCH_FAILED();
  }
  dca_launch(wls_solve_kernel<ROWS>, dim3(groups, L.S, B), WL, 0, st, U, V, w, (const float*)R, L, lam, final_pass,
             disp, pitch_row, pitch_img, min_support);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

}  // namespace dca

using namespace dca;

extern "C" int dca_wls_filter(const float* disp, const float* peak, const unsigned char* label, long long pitch_row,
                              long long pitch_img, int B, int H, int W, const unsigned char* guide, int channels,
                              long long guide_pitch_row, long long guide_pitch_img, const float* lut, float lambda,
                              int num_iter, float min_support, float* refined, float* support, void* workspace,
                              void* stream) {
  if (!disp || !guide || !lut || !refined || !support || !workspace) return DCA_ERR_ARG;
  if (B <= 0 || B > 65535 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  if (channels != 3 && channels != 4) return DCA_ERR_ARG;
  if (pitch_row < W || pitch_img < (long long)H * pitch_row) return DCA_ERR_ARG;
  if (guide_pitch_row < (long long)W * channels || guide_pitch_img < (long long)H * guide_pitch_row) return DCA_ERR_ARG;
  if (num_iter < 1 || num_iter > DCA_WLS_MAX_ITER) return DCA_ERR_ARG;
  if (!(lambda >= 0.f) || isinf(lambda) || !(min_support >= 0.f)) return DCA_ERR_ARG;     // NaN fails >= 0
  if ((long long)H * W > INT_MAX) return DCA_ERR_UNSUPPORTED;
  const WlsLines rows = {W, H, DCA_WLS_SEGMENTS(W), (long long)H * W, W, 1};
  const WlsLines cols = {H, W, DCA_WLS_SEGMENTS(H), (long long)H * W, 1, W};
  if (rows.S > 65535 || cols.S > 65535) return DCA_ERR_UNSUPPORTED;
  const size_t N = (size_t)B * H * W;
  float* ws = static_cast<float*>(workspace);
  float *wh = ws, *wv = ws + N, *Rr = ws + 2 * N, *Rc = Rr + (size_t)8 * B * H * rows.S;
  const cudaStream_t st = (cudaStream_t)stream;
  dca_launch(wls_prepare_kernel, dim3((unsigned)(((long long)H * W + WP_THREADS - 1) / WP_THREADS), B), WP_THREADS, 0,
             st, disp, peak, label, pitch_row, pitch_img, H, W, guide, channels, guide_pitch_row, guide_pitch_img, lut,
             refined, support, wh, wv);
  DCA_RETURN_IF_LAUNCH_FAILED();
  const double den = ldexp(1.0, 2 * num_iter) - 1.0;
  for (int t = 1; t <= num_iter; ++t) {
    const float lam = (float)((((double)lambda * 1.5) * ldexp(1.0, 2 * (num_iter - t))) / den);
    int rc = wls_pass<true>(refined, support, wh, Rr, rows, lam, 0, disp, pitch_row, pitch_img, min_support, B, st);
    if (rc != DCA_OK) return rc;
    rc = wls_pass<false>(refined, support, wv, Rc, cols, lam, t == num_iter ? 1 : 0, disp, pitch_row, pitch_img,
                         min_support, B, st);
    if (rc != DCA_OK) return rc;
  }
  return DCA_OK;
}
