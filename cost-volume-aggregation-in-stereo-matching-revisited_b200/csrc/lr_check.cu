// Left-right consistency check of a disparity pair and the background fill of the pixels that fail it.  Definitions:
// include/dca_b200.h section (8).
//
// One CTA per (image, row).  The D_L and D_R rows are staged in shared memory with coalesced loads (D_R read back to
// front when it is in the layout of the mirrored forward, so no flipped copy is ever materialised; the un-mirrored row
// is written to disp_right_out on the way when asked).  Labels are computed pixel-strided and written coalesced.  The
// nearest consistent index on each side comes from two block scans over thread-contiguous segments: a max-scan of the
// index from the left and a min-scan from the right, each a warp shuffle scan plus one cross-warp step over the warp
// totals.  The filled row replaces D_R in shared memory and leaves coalesced.
#include "dca_common.cuh"
#include "../../include/dca_b200.h"

namespace dca {

constexpr int LR_THREADS = 256;
constexpr int LR_WARPS = LR_THREADS / 32;
constexpr size_t LR_SMEM_PER_PIXEL = 2 * sizeof(float) + 1;      // D_L, D_R (later the filled row), label

// fp32 with explicit rounding, no contraction: a float32 numpy restatement reproduces it bit for bit
__device__ __forceinline__ unsigned char lr_label(float d, const float* s_dr, int x, int W, float tau) {
  const float xr = __fsub_rn(__int2float_rn(x), d);
  if (!(xr >= 0.f && xr <= __int2float_rn(W - 1))) return DCA_LR_OUT_OF_VIEW;     // NaN / inf d included
  const float x0f = floorf(xr);
  const int x0 = (int)x0f;
  const float r0 = s_dr[x0];
  const float v = x0 == W - 1 ? r0 : __fadd_rn(r0, __fmul_rn(__fsub_rn(xr, x0f), __fsub_rn(s_dr[x0 + 1], r0)));
  if (fabsf(__fsub_rn(d, v)) <= tau) return DCA_LR_CONSISTENT;
  if (__fsub_rn(v, d) > tau) return DCA_LR_OCCLUDED;
  return DCA_LR_MISMATCH;                                                          // NaN v included
}

__global__ void __launch_bounds__(LR_THREADS)
lr_consistency_kernel(const float* __restrict__ dl, const float* __restrict__ dr, int mirrored,
                      unsigned char* __restrict__ label, float* __restrict__ filled, float* __restrict__ dr_out, int H,
                      int W, float tau) {
  extern __shared__ float lr_smem[];
  float* s_dl = lr_smem;
  float* s_dr = lr_smem + W;                                   // D_R, then the filled row
  unsigned char* s_lab = reinterpret_cast<unsigned char*>(lr_smem + 2 * W);
  __shared__ int s_wl[LR_WARPS], s_wr[LR_WARPS];
  const size_t o = ((size_t)blockIdx.y * H + blockIdx.x) * W;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  pdl_wait();
  for (int x = t; x < W; x += LR_THREADS) {
    s_dl[x] = dl[o + x];
    const float r = dr[o + (mirrored ? W - 1 - x : x)];
    s_dr[x] = r;
    if (dr_out) dr_out[o + x] = r;
  }
  __syncthreads();
  for (int x = t; x < W; x += LR_THREADS) {
    const unsigned char c = lr_label(s_dl[x], s_dr, x, W, tau);
    s_lab[x] = c;
    label[o + x] = c;
  }
  __syncthreads();

  // thread t owns the segment [x0, x1); last / first consistent index in it (-1 / W: none)
  const int seg = (W + LR_THREADS - 1) / LR_THREADS;
  const int x0 = min(t * seg, W), x1 = min(x0 + seg, W);
  int last = -1, first = W;
  for (int x = x0; x < x1; ++x) {
    if (s_lab[x] == DCA_LR_CONSISTENT) {
      first = min(first, x);
      last = x;
    }
  }
  int incl_l = last, incl_r = first;          // inclusive max-scan from the left, min-scan from the right, in the warp
#pragma unroll
  for (int k = 1; k < 32; k <<= 1) {
    const int a = __shfl_up_sync(0xffffffffu, incl_l, k);
    const int b = __shfl_down_sync(0xffffffffu, incl_r, k);
    if (lane >= k) incl_l = max(incl_l, a);
    if (lane + k < 32) incl_r = min(incl_r, b);
  }
  if (lane == 31) s_wl[warp] = incl_l;
  if (lane == 0) s_wr[warp] = incl_r;
  int left = __shfl_up_sync(0xffffffffu, incl_l, 1);             // exclusive: the segments strictly left / right
  int right = __shfl_down_sync(0xffffffffu, incl_r, 1);
  if (lane == 0) left = -1;
  if (lane == 31) right = W;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < LR_WARPS; ++w) {
    if (w < warp) left = max(left, s_wl[w]);
    if (w > warp) right = min(right, s_wr[w]);
  }

  int l = left, r = x0;                       // r: nearest consistent index >= x inside the segment, x1 = none there
  for (int x = x0; x < x1; ++x) {
    const float d = s_dl[x];
    float f;
    if (s_lab[x] == DCA_LR_CONSISTENT) {
      l = x;
      f = d;
    } else {
      if (r <= x) {
        r = x + 1;
        while (r < x1 && s_lab[r] != DCA_LR_CONSISTENT) ++r;
      }
      const int rr = r < x1 ? r : right;
      if (l >= 0 && rr < W) f = fminf(s_dl[l], s_dl[rr]);
      else if (l >= 0) f = s_dl[l];
      else if (rr < W) f = s_dl[rr];
      else f = d;
    }
    s_dr[x] = f;                              // D_R is no longer read: every label is in s_lab
  }
  __syncthreads();
  for (int x = t; x < W; x += LR_THREADS) filled[o + x] = s_dr[x];
}

}  // namespace dca

using namespace dca;

extern "C" int dca_lr_consistency(const float* disp_left, const float* disp_right, int right_mirrored,
                                  unsigned char* label, float* filled, float* disp_right_out, int B, int H, int W,
                                  float tau, void* stream) {
  if (!disp_left || !disp_right || !label || !filled || B <= 0 || H <= 0 || W <= 0 || B > 65535 || !(tau >= 0.f))
    return DCA_ERR_ARG;
  if (W > DCA_LR_MAX_W) return DCA_ERR_UNSUPPORTED;
  dca_launch(lr_consistency_kernel, dim3(H, B), LR_THREADS, LR_SMEM_PER_PIXEL * W, (cudaStream_t)stream, disp_left,
             disp_right, right_mirrored != 0, label, filled, disp_right_out, H, W, tau);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
