// Rectification of raw uint8 stereo pairs and the standardised, framed network input.  Definitions: include/dca_b200.h
// section (10).
//
//   rectify_kernel        grid (tiles, 2 views, B), one CTA per tile of DCA_RECTIFY_TILE rectified pixels in row-major
//                         order, thread t handles pixels k * RT_THREADS + t.  Per pixel: the source coordinate from the
//                         map, four taps x three channels of bilinear interpolation, rounding to uint8, the HWC store.
//                         Per channel, the CTA's sums of q and q^2 are reduced in 32 bits (<= TILE * 255^2 < 2^32) and
//                         added to the image's 64-bit counters with one integer atomic each: the totals do not depend
//                         on the order of the atomics.
//   standardise_kernel    grid (tiles of the frame, 2 views, B).  The output of a channel depends on q alone, so every
//                         CTA first turns the image's moments into mean / std (fp64) and a 3 x 256 table of the fp32
//                         outputs, then writes each frame pixel from the table (0 outside the copy window).
#include <limits.h>

#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int RT_THREADS = 256;
constexpr int RT_WARPS = RT_THREADS / 32;
constexpr int RT_PER_THREAD = DCA_RECTIFY_TILE / RT_THREADS;
static_assert(RT_PER_THREAD * RT_THREADS == DCA_RECTIFY_TILE, "tile = whole passes of the block");
static_assert((unsigned long long)DCA_RECTIFY_TILE * 255u * 255u < (1ull << 32), "32-bit CTA sums of q^2");

// one channel: v = (1-ay)((1-ax) p00 + ax p01) + ay((1-ax) p10 + ax p11), no contraction, then round and clamp
__device__ __forceinline__ int bilerp_u8(float wx0, float ax, float wy0, float ay, float p00, float p01, float p10,
                                         float p11) {
  const float top = __fadd_rn(__fmul_rn(wx0, p00), __fmul_rn(ax, p01));
  const float bot = __fadd_rn(__fmul_rn(wx0, p10), __fmul_rn(ax, p11));
  const float v = __fadd_rn(__fmul_rn(wy0, top), __fmul_rn(ay, bot));
  return min(max(__float2int_rn(v), 0), 255);
}

__global__ void __launch_bounds__(RT_THREADS)
rectify_kernel(const unsigned char* __restrict__ left, const unsigned char* __restrict__ right, int C,
               long long pitch_row, long long pitch_img, int Hs, int Ws, const float2* __restrict__ maps, int H, int W,
               unsigned char* __restrict__ rgb, unsigned long long* __restrict__ moments) {
  __shared__ unsigned s_sum[RT_WARPS][6];
  const int view = blockIdx.y, b = blockIdx.z, t = threadIdx.x;
  const int HW = H * W;
  const unsigned char* src = (view ? right : left) + (size_t)b * pitch_img;
  const float2* map = maps + (size_t)view * HW;
  unsigned char* out = rgb + ((size_t)b * 2 + view) * HW * 3;
  const float wsf = (float)Ws, hsf = (float)Hs;          // exact: Ws, Hs <= 2^24
  pdl_wait();
  unsigned s[3] = {0u, 0u, 0u}, ss[3] = {0u, 0u, 0u};
#pragma unroll
  for (int k = 0; k < RT_PER_THREAD; ++k) {
    const unsigned p = blockIdx.x * DCA_RECTIFY_TILE + k * RT_THREADS + t;     // < 2^31 + TILE
    if (p >= (unsigned)HW) continue;
    const float2 m = __ldg(map + p);
    int q[3] = {0, 0, 0};
    // a coordinate outside (-1, Ws) x (-1, Hs), a non-finite one included, has all four taps outside the image or
    // weighted by an exact 0, so v = 0: skipping it gives the same q
    if (m.x > -1.f && m.x < wsf && m.y > -1.f && m.y < hsf) {
      const float fx = floorf(m.x), fy = floorf(m.y);
      const int x0 = (int)fx, y0 = (int)fy;
      const float ax = __fsub_rn(m.x, fx), ay = __fsub_rn(m.y, fy);
      const float wx0 = __fsub_rn(1.f, ax), wy0 = __fsub_rn(1.f, ay);
      const bool in_x0 = x0 >= 0, in_x1 = x0 + 1 < Ws, in_y0 = y0 >= 0, in_y1 = y0 + 1 < Hs;
      const unsigned char* r0 = src + (long long)y0 * pitch_row + (long long)x0 * C;
      const unsigned char* r1 = r0 + pitch_row;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float p00 = (in_y0 && in_x0) ? (float)__ldg(r0 + c) : 0.f;
        const float p01 = (in_y0 && in_x1) ? (float)__ldg(r0 + C + c) : 0.f;
        const float p10 = (in_y1 && in_x0) ? (float)__ldg(r1 + c) : 0.f;
        const float p11 = (in_y1 && in_x1) ? (float)__ldg(r1 + C + c) : 0.f;
        q[c] = bilerp_u8(wx0, ax, wy0, ay, p00, p01, p10, p11);
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      out[(size_t)p * 3 + c] = (unsigned char)q[c];
      s[c] += (unsigned)q[c];
      ss[c] += (unsigned)(q[c] * q[c]);
    }
  }
  const int lane = t & 31, warp = t >> 5;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const unsigned a = __reduce_add_sync(0xffffffffu, s[c]), a2 = __reduce_add_sync(0xffffffffu, ss[c]);
    if (lane == 0) {
      s_sum[warp][2 * c] = a;
      s_sum[warp][2 * c + 1] = a2;
    }
  }
  __syncthreads();
  if (t < 6) {
    unsigned v = 0u;
#pragma unroll
    for (int w = 0; w < RT_WARPS; ++w) v += s_sum[w][t];
    if (v) atomicAdd(moments + ((size_t)b * 2 + view) * 6 + t, (unsigned long long)v);
  }
}

// correctly rounded double of a non-negative 128-bit integer: the top 64 significant bits with the rest folded into a
// sticky bit 0 round to the same 53 bits as the whole value; the scaling by 2^s is exact
__device__ __forceinline__ double u128_to_double_rn(unsigned __int128 v) {
  const unsigned long long hi = (unsigned long long)(v >> 64), lo = (unsigned long long)v;
  if (hi == 0ull) return __ull2double_rn(lo);
  const int s = 64 - __clzll((long long)hi);
  const unsigned __int128 rest = v & (((unsigned __int128)1 << s) - 1);
  const unsigned long long top = (unsigned long long)(v >> s) | (rest != 0 ? 1ull : 0ull);
  return ldexp(__ull2double_rn(top), s);
}

__global__ void __launch_bounds__(RT_THREADS)
standardise_kernel(const unsigned char* __restrict__ rgb, const unsigned long long* __restrict__ moments, int H, int W,
                   float* __restrict__ out_left, float* __restrict__ out_right, int Hn, int Wn, int dst_y0, int src_y0,
                   int win_h, int win_w) {
  __shared__ double s_stat[3][2];
  __shared__ float s_lut[3][256];
  const int view = blockIdx.y, b = blockIdx.z, t = threadIdx.x;
  const int HWn = Hn * Wn;
  pdl_wait();
  if (t < 3) {
    const unsigned long long S = moments[((size_t)b * 2 + view) * 6 + 2 * t];
    const unsigned long long SS = moments[((size_t)b * 2 + view) * 6 + 2 * t + 1];
    const unsigned long long N = (unsigned long long)H * W;
    const unsigned __int128 num = (unsigned __int128)N * SS - (unsigned __int128)S * S;     // >= 0 (Cauchy-Schwarz)
    const double nd = __ull2double_rn(N);
    s_stat[t][0] = __ddiv_rn(__ull2double_rn(S), nd);
    s_stat[t][1] = __dsqrt_rn(__ddiv_rn(u128_to_double_rn(num), __dmul_rn(nd, nd)));
  }
  __syncthreads();
#pragma unroll
  for (int c = 0; c < 3; ++c)
    s_lut[c][t] = __double2float_rn(__ddiv_rn(__dsub_rn((double)t, s_stat[c][0]), s_stat[c][1]));
  __syncthreads();
  const unsigned char* img = rgb + ((size_t)b * 2 + view) * ((size_t)H * W * 3);
  float* out = (view ? out_right : out_left) + (size_t)b * 3 * HWn;
#pragma unroll
  for (int k = 0; k < RT_PER_THREAD; ++k) {
    const unsigned p = blockIdx.x * DCA_RECTIFY_TILE + k * RT_THREADS + t;
    if (p >= (unsigned)HWn) continue;
    const int yn = (int)p / Wn, xn = (int)p - yn * Wn;
    const int y = yn - dst_y0;
    float v[3] = {0.f, 0.f, 0.f};
    if (y >= 0 && y < win_h && xn < win_w) {
      const unsigned char* q = img + ((size_t)(y + src_y0) * W + xn) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = s_lut[c][q[c]];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) out[(size_t)c * HWn + p] = v[c];
  }
}

}  // namespace dca

using namespace dca;

extern "C" int dca_rectify(const unsigned char* left, const unsigned char* right, int channels, long long pitch_row,
                           long long pitch_img, int B, int Hs, int Ws, const float* maps, int H, int W,
                           unsigned char* rgb, unsigned long long* moments, void* stream) {
  if (!left || !right || !maps || !rgb || !moments) return DCA_ERR_ARG;
  if (B <= 0 || B > 65535 || Hs <= 0 || Ws <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  if (channels != 3 && channels != 4) return DCA_ERR_ARG;
  if (pitch_row < (long long)Ws * channels || pitch_img < (long long)Hs * pitch_row) return DCA_ERR_ARG;
  if ((long long)H * W > INT_MAX || (long long)Hs * Ws > INT_MAX || Hs > (1 << 24) || Ws > (1 << 24))
    return DCA_ERR_UNSUPPORTED;
  const int tiles = (int)(((long long)H * W + DCA_RECTIFY_TILE - 1) / DCA_RECTIFY_TILE);
  dca_launch(rectify_kernel, dim3(tiles, 2, B), RT_THREADS, 0, (cudaStream_t)stream, left, right, channels, pitch_row,
             pitch_img, Hs, Ws, reinterpret_cast<const float2*>(maps), H, W, rgb, moments);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_standardise_frame(const unsigned char* rgb, const unsigned long long* moments, int B, int H, int W,
                                     float* left, float* right, int Hn, int Wn, int dst_y0, int src_y0, int win_h,
                                     int win_w, void* stream) {
  if (!rgb || !moments || !left || !right) return DCA_ERR_ARG;
  if (B <= 0 || B > 65535 || H <= 0 || W <= 0 || Hn <= 0 || Wn <= 0 || win_h <= 0 || win_w <= 0) return DCA_ERR_ARG;
  if (dst_y0 < 0 || src_y0 < 0 || (long long)dst_y0 + win_h > Hn || (long long)src_y0 + win_h > H || win_w > Wn ||
      win_w > W)
    return DCA_ERR_ARG;
  if ((long long)H * W > INT_MAX || (long long)Hn * Wn > INT_MAX) return DCA_ERR_UNSUPPORTED;
  const int tiles = (int)(((long long)Hn * Wn + DCA_RECTIFY_TILE - 1) / DCA_RECTIFY_TILE);
  dca_launch(standardise_kernel, dim3(tiles, 2, B), RT_THREADS, 0, (cudaStream_t)stream, rgb, moments, H, W, left,
             right, Hn, Wn, dst_y0, src_y0, win_h, win_w);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
