// DCA-module kernels and the bandwidth-bound tail of the hot path (SURVEY 8a rows a4-pool, a6, a7,
// a8, a11, a12-upsample) plus layout / weight-packing utilities.
//
//   avgpool3d            nn.AvgPool3d(3, 2, 1)                       models/augment/cva.py:39
//   class_stats          softmax/argmax/per-class sums               models/augment/semantic_level.py:98-119
//   disp_attention       key scaling + q/k/v projections + 4-head attention over disparity + out
//                        projection (+ the aug half of cva.fuse)     semantic_level.py:126,
//                                                                    SelfAttention_bn.py:62-98, cva.py:55,69
//   upsample_fuse        trilinear x2 + cat + 1x1x1 fuse conv + BN    cva.py:64,69
//   softmax_regress      F.softmax(dim=1) + disparity_regression      gwcnet_dca_g.py:238-239, submodule.py:127-131
//   convex_upsample      PropgationNet_4x.forward tail                gwcnet_dca_g.py:118-124
#include "dca_common.cuh"
#include "class_argmax.cuh"

namespace dca {

// ------------------------------------------------------------------------------------------------
// AvgPool3d k3 s2 p1, count_include_pad=True (always /27).  thread = (output voxel, 8-channel chunk)
// ------------------------------------------------------------------------------------------------
template <int PLANES>
__global__ void __launch_bounds__(256)
avgpool3d_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int C, int Di, int Hi,
                 int Wi, int Do, int Ho, int Wo) {
  const int c8n = C / 8;
  const size_t total = (size_t)B * Do * Ho * Wo * c8n;
  const size_t xin_plane = (size_t)B * Di * Hi * Wi * C, yout_plane = (size_t)B * Do * Ho * Wo * C;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int c8 = (int)(i % c8n);
    size_t r = i / c8n;
    int ow = (int)(r % Wo); r /= Wo;
    int oh = (int)(r % Ho); r /= Ho;
    int od = (int)(r % Do);
    int b = (int)(r / Do);
    // packed fp32x2 adds (sm_100 FADD2): the kernel is issue bound on the bf16 unpack + accumulate stream
    float2 acc2[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) acc2[k] = make_float2(0.f, 0.f);
    for (int dz = -1; dz <= 1; ++dz) {
      int iz = 2 * od + dz;
      if (iz < 0 || iz >= Di) continue;
      for (int dy = -1; dy <= 1; ++dy) {
        int iy = 2 * oh + dy;
        if (iy < 0 || iy >= Hi) continue;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
          int ix = 2 * ow + dx;
          if (ix < 0 || ix >= Wi) continue;
          const size_t off = ((((size_t)b * Di + iz) * Hi + iy) * Wi + ix) * C + c8 * 8;
          const uint4 hv = *reinterpret_cast<const uint4*>(x + off);
          float f[8];
          unpack8(hv, f);
#pragma unroll
          for (int k = 0; k < 4; ++k) acc2[k] = __fadd2_rn(acc2[k], make_float2(f[2 * k], f[2 * k + 1]));
          if (PLANES == 2) {
            const uint4 lv = *reinterpret_cast<const uint4*>(x + xin_plane + off);
            unpack8(lv, f);
#pragma unroll
            for (int k = 0; k < 4; ++k) acc2[k] = __fadd2_rn(acc2[k], make_float2(f[2 * k], f[2 * k + 1]));
          }
        }
      }
    }
    float acc[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) { acc[2 * k] = acc2[k].x * (1.0f / 27.0f); acc[2 * k + 1] = acc2[k].y * (1.0f / 27.0f); }
    store8<PLANES>(y, yout_plane, ((((size_t)b * Do + od) * Ho + oh) * Wo + ow) * C + c8 * 8, acc);
  }
}

// ------------------------------------------------------------------------------------------------
// class statistics: P = softmax_d(logits); k_p = first argmax_d P; e_p = exp(P[k_p]); S[b,k] += e_p
// logits fp32 [B,D,H,W].  thread = pixel (coalesced along w for every d).
// ------------------------------------------------------------------------------------------------
constexpr int CS_MAXD = 256;
// S[b,k] is summed in 2^-40 FIXED POINT (64-bit integer atomics, shared then global): integer addition is associative, so
// the result does not depend on the order in which pixels / CTAs arrive -- two runs of the same forward are bit-identical
// (a float atomicAdd version differed in the last bit from run to run).  e_p = exp(P[k_p]) lies in (1, e], sums stay
// below 2^58 for any image the path can hold.  The last CTA to finish (ticket) converts the sums to fp32.
constexpr float CS_FIX = 1099511627776.0f;   // 2^40
// The per-pixel softmax / first argmax (pixel_class_stats) lives in class_argmax.cuh, shared with dca_class_confusion.

// fixed-point per-class sums of one warp of pixels: summed per class inside the warp, one atomic per (warp, class)
__device__ __forceinline__ void warp_class_sums(unsigned long long* dst, int lane, int kk, unsigned long long efix) {
  unsigned todo = __ballot_sync(0xffffffffu, kk >= 0);
  while (todo) {
    const int leader = __ffs(todo) - 1;
    const int k0 = __shfl_sync(0xffffffffu, kk, leader);
    const bool mine = (kk == k0);
    unsigned long long v = mine ? efix : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == leader) atomicAdd(&dst[k0], v);
    todo &= ~__ballot_sync(0xffffffffu, mine);
  }
}

__global__ void __launch_bounds__(CS_THREADS)
class_stats_kernel(const float* __restrict__ logits, int* __restrict__ cls, float* __restrict__ e_out,
                   float* __restrict__ S, unsigned long long* __restrict__ acc /* [B*D] sums + [1] ticket, zeroed */,
                   int D, int HW, int BD) {
  __shared__ CsSmem sm;
  __shared__ int s_last;
  pdl_wait();
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int p = blockIdx.x * 32 + lane;
  const bool valid = p < HW;
  const float* lp = logits + (size_t)b * D * HW + (valid ? p : 0);
  int k = 0;
  float e = 0.f;
  pixel_class_stats<0>(sm, lane, g, D, valid, [&](int d) { return __ldg(lp + (size_t)d * HW); }, k, e);
  if (g == 0) {
    if (valid) {
      cls[(size_t)b * HW + p] = k;
      e_out[(size_t)b * HW + p] = e;
    }
    warp_class_sums(acc + (size_t)b * D, lane, valid ? k : -1, valid ? __float2ull_rn(e * CS_FIX) : 0ull);
    __threadfence();
    if (lane == 0) {
      const unsigned long long t = atomicAdd(&acc[BD], 1ull);
      s_last = (t == (unsigned long long)gridDim.x * gridDim.y - 1ull);
    }
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    for (int i = threadIdx.x; i < BD; i += blockDim.x) {
      const unsigned long long v = *reinterpret_cast<volatile unsigned long long*>(&acc[i]);
      S[i] = (float)((double)v * (1.0 / 1099511627776.0));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Fused DCA attention.  One warp per pixel, lane = channel (C == 32 == 4 heads x 8).
//   key[d] = x[d] * (1 + [d == k_p] * e_p / S[b,k_p])
//   q = Pq1(Pq0(x)), k = Pk1(Pk0(key)), v = Pv(key);  P = 1x1x1 conv + BN + LeakyReLU(0.1)
//   ctx[dq, head] = softmax_dk(q[dq,head] . k[dk,head] / sqrt(8)) v[dk, head]
//   out = Po(ctx);  optional  t = Wa . out  (the aug half of cva.fuse, linear, commutes with the
//   trilinear upsampling that follows)
// Weights: 7 matrices stored transposed [ci][co] fp32, then 6 x (scale[32], shift[32]).
// ------------------------------------------------------------------------------------------------
constexpr int AT_C = 32;
__device__ __forceinline__ float fast_exp2(float x) {   // ex2.approx: rel. error 2^-22, -inf -> 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr int AT_NMAT = 7;
constexpr int AT_WFLOATS = AT_NMAT * AT_C * AT_C + 6 * 2 * AT_C;

// ---- warp-level tensor-core projection (mma.sync m16n8k16 bf16, fp32 accumulate, split-bf16 operands) ----
// Activations live in shared memory as two bf16 planes (hi, lo), rows of 32 channels padded to 40 elements
// (80 B pitch: conflict-free ldmatrix).  Weights are [co][ci] (K-major) bf16 hi/lo with the same pitch.
// y[d][co] = act(scale[co] * sum_ci x[d][ci] W[co][ci] + shift[co]),  x.W ~ hi.Whi + hi.Wlo + lo.Whi
constexpr int AT_PITCH = 40;                         // bf16 elements per smem row
constexpr int AT_WPLANE = AT_C * AT_PITCH;           // one weight plane (32 rows)

__device__ __forceinline__ void ldsm_x4(uint32_t saddr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
__device__ __forceinline__ void mma_bf16(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
#if DCA_F16_PLANES
#define DCA_MMA_TYPES "f16.f16"
#else
#define DCA_MMA_TYPES "bf16.bf16"
#endif
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32." DCA_MMA_TYPES ".f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
               "{%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void at_split2(float a, float b, uint32_t& hi, uint32_t& lo) { split_pair(a, b, hi, lo); }
__device__ __forceinline__ void ldsm_x4_trans(uint32_t saddr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
// m16n8k8: A = {a0 (rows 0-7), a1 (rows 8-15)}, B = {b0}
__device__ __forceinline__ void mma_k8(float* c, uint32_t a0, uint32_t a1, uint32_t b0) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32." DCA_MMA_TYPES ".f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(b0));
}

// src: bf16 pair [2][rows][AT_PITCH]; Wm: weight pair [2][32][AT_PITCH]; MT = number of 16-row tiles.
// dst_pair != nullptr: result written as a bf16 pair (input of the next projection);
// dst_f32  != nullptr: result written as fp32 [rows][32].
// MT = 16-row tiles this warp computes, starting at row0; ROWS = rows of the whole buffer (plane pitch).
template <int MT, int ROWS>
__device__ __forceinline__ void warp_project_mma(const __nv_bfloat16* __restrict__ src, const __nv_bfloat16* __restrict__ Wm,
                                                 const float* __restrict__ ss, bool affine_act,
                                                 __nv_bfloat16* __restrict__ dst_pair, float* __restrict__ dst_f32,
                                                 int lane, int row0 = 0) {
  float acc[MT][4][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
  const uint32_t s_src = (uint32_t)__cvta_generic_to_shared(src);
  const uint32_t s_w = (uint32_t)__cvta_generic_to_shared(Wm);
  // ldmatrix row address of this lane: A tiles (row = l%8 + 8*((l/8)%2), col = 8*(l/16)); B tiles (two n-tiles per x4:
  // row n = l%8 + 8*(l/16), col k = 8*((l/8)%2))
  const int a_row = (lane & 7) + ((lane >> 3) & 1) * 8, a_col = (lane >> 4) * 8;
  const int b_row = (lane & 7) + (lane >> 4) * 8, b_col = ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int kt = 0; kt < 2; ++kt) {
    uint32_t bh[4][2], bl[4][2];
#pragma unroll
    for (int np = 0; np < 2; ++np) {           // n-tile pairs (0,1) and (2,3)
      const uint32_t off = (uint32_t)(((np * 16 + b_row) * AT_PITCH + kt * 16 + b_col) * 2);
      ldsm_x4(s_w + off, bh[2 * np][0], bh[2 * np][1], bh[2 * np + 1][0], bh[2 * np + 1][1]);
      ldsm_x4(s_w + AT_WPLANE * 2 + off, bl[2 * np][0], bl[2 * np][1], bl[2 * np + 1][0], bl[2 * np + 1][1]);
    }
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      uint32_t ah[4], al[4];
      const uint32_t off = (uint32_t)(((row0 + mt * 16 + a_row) * AT_PITCH + kt * 16 + a_col) * 2);
      ldsm_x4(s_src + off, ah[0], ah[1], ah[2], ah[3]);
      ldsm_x4(s_src + ROWS * AT_PITCH * 2 + off, al[0], al[1], al[2], al[3]);
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        mma_bf16(acc[mt][nt], ah, bh[nt][0], bh[nt][1]);
        mma_bf16(acc[mt][nt], ah, bl[nt][0], bl[nt][1]);
        mma_bf16(acc[mt][nt], al, bh[nt][0], bh[nt][1]);
      }
    }
  }
  // epilogue: thread (g = lane/4, t = lane%4) holds rows g, g+8 and columns nt*8 + 2t, +1 of every tile
  const int g = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    const int col = nt * 8 + t2;
    float sc0 = 1.f, sc1 = 1.f, sh0 = 0.f, sh1 = 0.f;
    if (affine_act) { sc0 = ss[col]; sc1 = ss[col + 1]; sh0 = ss[AT_C + col]; sh1 = ss[AT_C + col + 1]; }
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int row = row0 + mt * 16 + g + hrow * 8;
        float v0 = acc[mt][nt][hrow * 2] * sc0 + sh0, v1 = acc[mt][nt][hrow * 2 + 1] * sc1 + sh1;
        if (affine_act) { v0 = v0 > 0.f ? v0 : 0.1f * v0; v1 = v1 > 0.f ? v1 : 0.1f * v1; }
        if (dst_f32) *reinterpret_cast<float2*>(dst_f32 + row * AT_C + col) = make_float2(v0, v1);
        if (dst_pair) {
          uint32_t hi, lo;
          at_split2(v0, v1, hi, lo);
          *reinterpret_cast<uint32_t*>(dst_pair + row * AT_PITCH + col) = hi;
          *reinterpret_cast<uint32_t*>(dst_pair + ROWS * AT_PITCH + row * AT_PITCH + col) = lo;
        }
      }
    }
  }
  __syncwarp();
}

// DT = compile-time disparity count (24 at KITTI/SceneFlow: scores stay in registers, two-pass softmax); 0 = runtime D
// WPP = warps per pixel: 1 = a warp walks a pixel alone; 2 = a TEAM of two warps shares a pixel's buffers (each computes
// 16 of the 32 projection rows, half of the attention items and half of the stores; phases are separated by a 64-thread
// named barrier), which doubles the resident warps for the same shared memory: the kernel is latency bound.
// CORE = 1 (team mode, D/8 == 24): the attention core itself also runs on mma.sync -- S = q k^T per head as m16n8k8
// tiles (3 split terms), softmax on the accumulator fragments, P V as m16n8k16 tiles with P re-split to hi/lo in
// registers -- instead of one fp32 FMA chain per (query, head) item with broadcast LDS.128 reads of k and v.
template <int PLANES, int MT, int DT, int WPP, int CORE>
__global__ void __launch_bounds__(CORE ? 576 : 256 * WPP)
disp_attention_kernel(const __nv_bfloat16* __restrict__ x, const int* __restrict__ cls, const float* __restrict__ e,
                      const float* __restrict__ S, const float* __restrict__ wts, int has_wa,
                      __nv_bfloat16* __restrict__ y, int B, int D, int H, int Wd, int pad,
                      const __nv_bfloat16* __restrict__ key_feats) {
  // key_feats != nullptr: the generic two-input form SelfAttentionBlock.forward(query_feats, key_feats)
  // (SelfAttention_bn.py:62-98): the key rows are read from their own tensor instead of being built from (cls, e, S)
  constexpr int ROWS = 16 * MT;
  constexpr int PAIR = 2 * ROWS * AT_PITCH;                    // bf16 elements of one (hi, lo) activation pair
  constexpr int FBUF = ROWS * AT_C;                            // floats of one fp32 buffer
  const int HW = H * Wd;
  extern __shared__ __align__(16) uint8_t smem_at[];
  __nv_bfloat16* Wsm = reinterpret_cast<__nv_bfloat16*>(smem_at);               // [7][2][32][AT_PITCH]
  float* ss = reinterpret_cast<float*>(smem_at + AT_NMAT * 2 * AT_WPLANE * 2);   // 6 x (scale[32], shift[32])
  static_assert(WPP == 1 || (WPP == 2 && MT == 2 && DT > 0), "team mode: 32 rows, compile-time D");
  static_assert(CORE == 0 || (WPP == 2 && DT == 24), "mma core: two warps x 16 query rows, 24 keys");
  constexpr int TEAM_BYTES = CORE ? 4 * PAIR * 2 : 2 * PAIR * 2 + 3 * FBUF * 4;
  const int lane = threadIdx.x & 31;
  const int warps = (blockDim.x >> 5) / WPP, warp = (threadIdx.x >> 5) / WPP;    // teams per CTA, this warp's team
  const int wip = (threadIdx.x >> 5) % WPP;                                      // warp index inside the team
  constexpr int MTW = MT / WPP;                                                  // projection tiles per warp
  const int row0 = wip * 16 * MTW;
  auto team_sync = [&]() {
    if (WPP == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + warp), "r"(32 * WPP) : "memory");
  };
  uint8_t* wbase = smem_at + AT_NMAT * 2 * AT_WPLANE * 2 + 6 * 64 * 4 + (size_t)warp * TEAM_BYTES;
  __nv_bfloat16* P0 = reinterpret_cast<__nv_bfloat16*>(wbase);     // x, then key (row k_p rescaled in place), then ctx
  __nv_bfloat16* P2 = P0 + PAIR;                                   // intermediate of the two-layer projections
  // CORE = 0: q, k, v as fp32 (F0, F1, F2).  CORE = 1: q, k as hi/lo pairs (Pq, Pk), v in P2 (free after the key
  // projections); the fp32 result buffer F0 then aliases Pq, which is dead once the core is done.
  __nv_bfloat16* Pq = P2 + PAIR;
  __nv_bfloat16* Pk = Pq + PAIR;
  float* F0 = reinterpret_cast<float*>(P2 + PAIR);
  float* F1 = F0 + FBUF;
  float* F2 = F1 + FBUF;
  // weights arrive fp32, transposed [m][ci][co]; keep them as bf16 hi/lo [m][plane][co][ci]
  for (int i = threadIdx.x; i < AT_NMAT * AT_C * AT_C; i += blockDim.x) {
    const int m = i >> 10, r = i & 1023, ci = r >> 5, co = r & 31;
    uint32_t lo;
    const uint32_t hi = split_bf16(__ldg(wts + i), lo);
    Wsm[(m * 2 + 0) * AT_WPLANE + co * AT_PITCH + ci] = __ushort_as_bfloat16((unsigned short)hi);
    Wsm[(m * 2 + 1) * AT_WPLANE + co * AT_PITCH + ci] = __ushort_as_bfloat16((unsigned short)lo);
  }
  for (int i = threadIdx.x; i < 6 * 64; i += blockDim.x) ss[i] = __ldg(wts + AT_NMAT * AT_C * AT_C + i);
  // zero this warp's buffers once: rows [D, ROWS) are never loaded and must stay finite
  for (int i = lane + 32 * wip; i < TEAM_BYTES / 4; i += 32 * WPP) reinterpret_cast<uint32_t*>(wbase)[i] = 0u;
  pdl_trigger();       // persistent single-wave grid; the weight staging above only read static data
  pdl_wait();
  __syncthreads();
  const __nv_bfloat16* Wq0 = Wsm, *Wq1 = Wsm + 2 * AT_WPLANE, *Wk0 = Wsm + 4 * AT_WPLANE, *Wk1 = Wsm + 6 * AT_WPLANE,
                      *Wv = Wsm + 8 * AT_WPLANE, *Wo = Wsm + 10 * AT_WPLANE, *Wa = Wsm + 12 * AT_WPLANE;
  const size_t plane = (size_t)B * D * HW * AT_C;
  const float qscale = 0.35355339059327373f * 1.4426950408889634f;   // 8^-0.5 * log2(e): scores in the log2 domain

  // CORE mode: the rows of the NEXT pixel (and its class / weight) are fetched into registers while this one is processed
  uint4 pf_h[2], pf_l[2];
  int pf_kp = 0;
  float pf_e = 0.f;
  auto prefetch = [&](int pixn) {
    if (pixn >= B * HW) return;
    const int bn = pixn / HW, pn = pixn % HW;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int d = 8 * wip + 16 * r + (lane >> 2);
      if (d < D) {
        const size_t off = (((size_t)bn * D + d) * HW + pn) * AT_C + (lane & 3) * 8;
        pf_h[r] = *reinterpret_cast<const uint4*>(x + off);
        pf_l[r] = (PLANES == 2) ? *reinterpret_cast<const uint4*>(x + plane + off) : make_uint4(0, 0, 0, 0);
      }
    }
    if (key_feats == nullptr) {
      pf_kp = cls[pixn];
      pf_e = e[pixn];
    }
  };
  if (CORE) prefetch(blockIdx.x * warps + warp);
  for (int pix = blockIdx.x * warps + warp; pix < B * HW; pix += gridDim.x * warps) {
    const int b = pix / HW, p = pix % HW;
    const int kp = key_feats ? -1 : (CORE ? pf_kp : cls[pix]);
    const float wp = key_feats ? 0.f : (CORE ? pf_e : e[pix]) / S[(size_t)b * D + kp];
    // ---- x (already hi/lo in HBM) -> P0 verbatim ----
    if (CORE) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int d = 8 * wip + 16 * r + (lane >> 2), q = lane & 3;
        if (d < D) {
          *reinterpret_cast<uint4*>(P0 + d * AT_PITCH + q * 8) = pf_h[r];
          *reinterpret_cast<uint4*>(P0 + ROWS * AT_PITCH + d * AT_PITCH + q * 8) = pf_l[r];
        }
      }
      prefetch(pix + gridDim.x * warps);
    } else
    for (int d0 = 8 * wip; d0 < D; d0 += 8 * WPP) {
      const int d = d0 + (lane >> 2), q = lane & 3;
      if (d < D) {
        const size_t off = (((size_t)b * D + d) * HW + p) * AT_C + q * 8;
        const uint4 h = *reinterpret_cast<const uint4*>(x + off);
        uint4 l = make_uint4(0, 0, 0, 0);
        if (PLANES == 2) l = *reinterpret_cast<const uint4*>(x + plane + off);
        *reinterpret_cast<uint4*>(P0 + d * AT_PITCH + q * 8) = h;
        *reinterpret_cast<uint4*>(P0 + ROWS * AT_PITCH + d * AT_PITCH + q * 8) = l;
      }
    }
    team_sync();
    // (projections are row-wise: a warp only ever reads the rows it wrote itself, so no team barrier in between)
    warp_project_mma<MTW, ROWS>(P0, Wq0, ss + 0 * 64, true, P2, nullptr, lane, row0);
    if (CORE) warp_project_mma<MTW, ROWS>(P2, Wq1, ss + 1 * 64, true, Pq, nullptr, lane, row0);   // q -> Pq (hi/lo)
    else warp_project_mma<MTW, ROWS>(P2, Wq1, ss + 1 * 64, true, nullptr, F0, lane, row0);        // q -> F0 (fp32)
    // key = x * (1 + [d == k_p] w_p): only row k_p differs from x, so it is rescaled (and re-split) in place by the warp
    // that owns the row; the query projections above were the last readers of the plain row
    if (kp >= row0 && kp < row0 + 16 * MTW && lane < 4) {
      __nv_bfloat16* rh = P0 + kp * AT_PITCH + lane * 8;
      __nv_bfloat16* rl = rh + ROWS * AT_PITCH;
      float f[8], g2[8];
      unpack8(*reinterpret_cast<const uint4*>(rh), f);
      unpack8(*reinterpret_cast<const uint4*>(rl), g2);
      const float ks = 1.f + wp;
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) at_split2((f[2 * j] + g2[2 * j]) * ks, (f[2 * j + 1] + g2[2 * j + 1]) * ks, hw[j], lw[j]);
      *reinterpret_cast<uint4*>(rh) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      *reinterpret_cast<uint4*>(rl) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
    if (key_feats != nullptr) {
      // explicit key tensor: this warp replaces ITS rows [row0, row0 + 16*MTW) of P0 (the only rows it reads below)
      for (int r0 = 0; r0 < 16 * MTW; r0 += 8) {
        const int d = row0 + r0 + (lane >> 2), q = lane & 3;
        if (d < D) {
          const size_t off = (((size_t)b * D + d) * HW + p) * AT_C + q * 8;
          *reinterpret_cast<uint4*>(P0 + d * AT_PITCH + q * 8) = *reinterpret_cast<const uint4*>(key_feats + off);
          *reinterpret_cast<uint4*>(P0 + ROWS * AT_PITCH + d * AT_PITCH + q * 8) =
              (PLANES == 2) ? *reinterpret_cast<const uint4*>(key_feats + plane + off) : make_uint4(0, 0, 0, 0);
        }
      }
    }
    __syncwarp();
    warp_project_mma<MTW, ROWS>(P0, Wk0, ss + 2 * 64, true, P2, nullptr, lane, row0);
    if (CORE) warp_project_mma<MTW, ROWS>(P2, Wk1, ss + 3 * 64, true, Pk, nullptr, lane, row0);   // k -> Pk
    else warp_project_mma<MTW, ROWS>(P2, Wk1, ss + 3 * 64, true, nullptr, F1, lane, row0);        // k -> F1
    if (CORE) warp_project_mma<MTW, ROWS>(P0, Wv, ss + 4 * 64, true, P2, nullptr, lane, row0);    // v -> P2
    else warp_project_mma<MTW, ROWS>(P0, Wv, ss + 4 * 64, true, nullptr, F2, lane, row0);         // v -> F2
    team_sync();
    // ---- attention: item = (dq, head), 4 heads x D queries; a lane owns up to 2*MT items and walks the keys ONCE
    //      for all of them (independent online-softmax chains interleave -> ILP); ctx -> P0 as a bf16 pair ----
    if (CORE) {
      // ---- tensor-core attention core: this warp owns query rows [row0, row0 + 16); keys 0..23 = three n-tiles ----
      const uint32_t s_q = (uint32_t)__cvta_generic_to_shared(Pq), s_k = (uint32_t)__cvta_generic_to_shared(Pk),
                     s_v = (uint32_t)__cvta_generic_to_shared(P2);
      constexpr uint32_t LO = (uint32_t)(ROWS * AT_PITCH * 2);       // byte offset of the lo plane
      const int g = lane >> 2, t2 = (lane & 3) * 2;
      const int mrow = lane & 7, mid = lane >> 3;                    // ldmatrix: lane -> (row in matrix, matrix index)
#pragma unroll 1
      for (int hd = 0; hd < 4; ++hd) {
        // A = q[row0 + 0..15][hd*8 .. +8): matrices (hi rows 0-7, hi rows 8-15, lo rows 0-7, lo rows 8-15)
        uint32_t qh0, qh1, ql0, ql1;
        ldsm_x4(s_q + (uint32_t)(((row0 + (mid & 1) * 8 + mrow) * AT_PITCH + hd * 8) * 2) + (mid >> 1) * LO, qh0, qh1, ql0, ql1);
        // B = k[key][hd*8 .. +8) for key blocks 0-7, 8-15, 16-23 (the 4th matrix, rows 24-31, is not used)
        uint32_t kh[4], kl[4];
        const uint32_t koff = (uint32_t)(((mid * 8 + mrow) * AT_PITCH + hd * 8) * 2);
        ldsm_x4(s_k + koff, kh[0], kh[1], kh[2], kh[3]);
        ldsm_x4(s_k + LO + koff, kl[0], kl[1], kl[2], kl[3]);
        float sc[3][4];
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
          sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
          mma_k8(sc[nt], qh0, qh1, kh[nt]);
          mma_k8(sc[nt], qh0, qh1, kl[nt]);
          mma_k8(sc[nt], ql0, ql1, kh[nt]);
        }
        // softmax over the 24 keys of rows g (values [nt][0..1]) and g + 8 ([nt][2..3]), log2 domain
        float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
#pragma unroll
          for (int i = 0; i < 4; ++i) sc[nt][i] *= qscale;
          m0 = fmaxf(m0, fmaxf(sc[nt][0], sc[nt][1]));
          m1 = fmaxf(m1, fmaxf(sc[nt][2], sc[nt][3]));
        }
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
        float l0 = 0.f, l1 = 0.f;
        uint32_t ph[3][2], pl[3][2];                                 // P as packed hi / lo pairs: [n-tile][row g / g+8]
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
          const float p0 = fast_exp2(sc[nt][0] - m0), p1 = fast_exp2(sc[nt][1] - m0);
          const float p2 = fast_exp2(sc[nt][2] - m1), p3 = fast_exp2(sc[nt][3] - m1);
          l0 += p0 + p1; l1 += p2 + p3;
          at_split2(p0, p1, ph[nt][0], pl[nt][0]);
          at_split2(p2, p3, ph[nt][1], pl[nt][1]);
        }
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        // B = v^T: transposed 8x8 blocks of v[key][hd*8 .. +8) for key blocks 0-7, 8-15, 16-23, 24-31 (finite padding)
        uint32_t vh[4], vl[4];
        ldsm_x4_trans(s_v + koff, vh[0], vh[1], vh[2], vh[3]);
        ldsm_x4_trans(s_v + LO + koff, vl[0], vl[1], vl[2], vl[3]);
        float cx[4] = {0.f, 0.f, 0.f, 0.f};
        {
          const uint32_t a_hi[4] = {ph[0][0], ph[0][1], ph[1][0], ph[1][1]}, a_lo[4] = {pl[0][0], pl[0][1], pl[1][0], pl[1][1]};
          mma_bf16(cx, a_hi, vh[0], vh[1]);
          mma_bf16(cx, a_hi, vl[0], vl[1]);
          mma_bf16(cx, a_lo, vh[0], vh[1]);
          const uint32_t b_hi[4] = {ph[2][0], ph[2][1], 0u, 0u}, b_lo[4] = {pl[2][0], pl[2][1], 0u, 0u};
          mma_bf16(cx, b_hi, vh[2], vh[3]);
          mma_bf16(cx, b_hi, vl[2], vl[3]);
          mma_bf16(cx, b_lo, vh[2], vh[3]);
        }
        const float i0 = 1.f / l0, i1 = 1.f / l1;
        uint32_t h0, lo0, h1, lo1;
        at_split2(cx[0] * i0, cx[1] * i0, h0, lo0);
        at_split2(cx[2] * i1, cx[3] * i1, h1, lo1);
        __nv_bfloat16* c0p = P0 + (row0 + g) * AT_PITCH + hd * 8 + t2;
        *reinterpret_cast<uint32_t*>(c0p) = h0;
        *reinterpret_cast<uint32_t*>(c0p + ROWS * AT_PITCH) = lo0;
        *reinterpret_cast<uint32_t*>(c0p + 8 * AT_PITCH) = h1;
        *reinterpret_cast<uint32_t*>(c0p + 8 * AT_PITCH + ROWS * AT_PITCH) = lo1;
      }
    } else
    if (DT > 0) {
      // scores of a lane's items stay in registers: pass 1 = all dot products + running max, pass 2 = exp2 and P.V
      constexpr int NI = (4 * (DT > 0 ? DT : 1) + 32 * WPP - 1) / (32 * WPP);
      constexpr int DK = DT > 0 ? DT : 1;
      // item = (dq, head) = ((lane + 32 r) * WPP + wip): a team splits the items by parity
      const int hd = (lane * WPP + wip) & 3;
      float sc[NI][DK], mx[NI];
      {
        float4 qa[NI], qb[NI];
#pragma unroll
        for (int r = 0; r < NI; ++r) {
          const int dq = min(((lane + 32 * r) * WPP + wip) >> 2, ROWS - 1);
          qa[r] = *reinterpret_cast<const float4*>(F0 + dq * AT_C + hd * 8);
          qb[r] = *reinterpret_cast<const float4*>(F0 + dq * AT_C + hd * 8 + 4);
          qa[r].x *= qscale; qa[r].y *= qscale; qa[r].z *= qscale; qa[r].w *= qscale;
          qb[r].x *= qscale; qb[r].y *= qscale; qb[r].z *= qscale; qb[r].w *= qscale;
          mx[r] = -INFINITY;
        }
#pragma unroll
        for (int dk = 0; dk < DK; ++dk) {
          const float4 k0 = *reinterpret_cast<const float4*>(F1 + dk * AT_C + hd * 8);
          const float4 k1 = *reinterpret_cast<const float4*>(F1 + dk * AT_C + hd * 8 + 4);
#pragma unroll
          for (int r = 0; r < NI; ++r) {
            sc[r][dk] = (qa[r].x * k0.x + qa[r].y * k0.y) + (qa[r].z * k0.z + qa[r].w * k0.w) +
                        (qb[r].x * k1.x + qb[r].y * k1.y) + (qb[r].z * k1.z + qb[r].w * k1.w);
            mx[r] = fmaxf(mx[r], sc[r][dk]);
          }
        }
      }
      float ls[NI], c[NI][8];
#pragma unroll
      for (int r = 0; r < NI; ++r) {
        ls[r] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) c[r][i] = 0.f;
      }
#pragma unroll
      for (int dk = 0; dk < DK; ++dk) {
        const float4 v0 = *reinterpret_cast<const float4*>(F2 + dk * AT_C + hd * 8);
        const float4 v1 = *reinterpret_cast<const float4*>(F2 + dk * AT_C + hd * 8 + 4);
#pragma unroll
        for (int r = 0; r < NI; ++r) {
          const float pe = fast_exp2(sc[r][dk] - mx[r]);
          ls[r] += pe;
          c[r][0] = fmaf(pe, v0.x, c[r][0]); c[r][1] = fmaf(pe, v0.y, c[r][1]);
          c[r][2] = fmaf(pe, v0.z, c[r][2]); c[r][3] = fmaf(pe, v0.w, c[r][3]);
          c[r][4] = fmaf(pe, v1.x, c[r][4]); c[r][5] = fmaf(pe, v1.y, c[r][5]);
          c[r][6] = fmaf(pe, v1.z, c[r][6]); c[r][7] = fmaf(pe, v1.w, c[r][7]);
        }
      }
#pragma unroll
      for (int r = 0; r < NI; ++r) {
        const int item = (lane + 32 * r) * WPP + wip;
        if (item < 4 * D) {
          const int dq = item >> 2;
          const float il = 1.f / ls[r];
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) at_split2(c[r][2 * j] * il, c[r][2 * j + 1] * il, hw[j], lw[j]);
          *reinterpret_cast<uint4*>(P0 + dq * AT_PITCH + hd * 8) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(P0 + ROWS * AT_PITCH + dq * AT_PITCH + hd * 8) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
    } else
    {
      constexpr int NI = 2 * MT;
      float4 qa[NI], qb[NI];
      float mx[NI], ls[NI], c[NI][8];
      int hdv[NI];
#pragma unroll
      for (int r = 0; r < NI; ++r) {
        const int item = lane + 32 * r;
        const int dq = min(item >> 2, ROWS - 1);
        hdv[r] = item & 3;
        qa[r] = *reinterpret_cast<const float4*>(F0 + dq * AT_C + hdv[r] * 8);
        qb[r] = *reinterpret_cast<const float4*>(F0 + dq * AT_C + hdv[r] * 8 + 4);
        qa[r].x *= qscale; qa[r].y *= qscale; qa[r].z *= qscale; qa[r].w *= qscale;
        qb[r].x *= qscale; qb[r].y *= qscale; qb[r].z *= qscale; qb[r].w *= qscale;
        mx[r] = -INFINITY; ls[r] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) c[r][i] = 0.f;
      }
      const int hd = lane & 3;                     // item & 3 == lane & 3 for every r
      for (int dk = 0; dk < D; ++dk) {
        const float4 k0 = *reinterpret_cast<const float4*>(F1 + dk * AT_C + hd * 8);
        const float4 k1 = *reinterpret_cast<const float4*>(F1 + dk * AT_C + hd * 8 + 4);
        const float4 v0 = *reinterpret_cast<const float4*>(F2 + dk * AT_C + hd * 8);
        const float4 v1 = *reinterpret_cast<const float4*>(F2 + dk * AT_C + hd * 8 + 4);
#pragma unroll
        for (int r = 0; r < NI; ++r) {
          const float s2 = (qa[r].x * k0.x + qa[r].y * k0.y) + (qa[r].z * k0.z + qa[r].w * k0.w) +
                           (qb[r].x * k1.x + qb[r].y * k1.y) + (qb[r].z * k1.z + qb[r].w * k1.w);
          const float mn = fmaxf(mx[r], s2);
          const float corr = fast_exp2(mx[r] - mn), pe = fast_exp2(s2 - mn);
          ls[r] = ls[r] * corr + pe;
          c[r][0] = c[r][0] * corr + pe * v0.x; c[r][1] = c[r][1] * corr + pe * v0.y;
          c[r][2] = c[r][2] * corr + pe * v0.z; c[r][3] = c[r][3] * corr + pe * v0.w;
          c[r][4] = c[r][4] * corr + pe * v1.x; c[r][5] = c[r][5] * corr + pe * v1.y;
          c[r][6] = c[r][6] * corr + pe * v1.z; c[r][7] = c[r][7] * corr + pe * v1.w;
          mx[r] = mn;
        }
      }
#pragma unroll
      for (int r = 0; r < NI; ++r) {
        const int item = lane + 32 * r;
        if (item < 4 * D) {
          const int dq = item >> 2;
          const float il = 1.f / ls[r];
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) at_split2(c[r][2 * j] * il, c[r][2 * j + 1] * il, hw[j], lw[j]);
          *reinterpret_cast<uint4*>(P0 + dq * AT_PITCH + hd * 8) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(P0 + ROWS * AT_PITCH + dq * AT_PITCH + hd * 8) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
    }
    team_sync();
    const float* res;
    if (has_wa) {
      warp_project_mma<MTW, ROWS>(P0, Wo, ss + 5 * 64, true, P2, nullptr, lane, row0);    // aug_down -> P2
      warp_project_mma<MTW, ROWS>(P2, Wa, nullptr, false, nullptr, F0, lane, row0);       // t = Wa . aug_down -> F0
      res = F0;
    } else {
      warp_project_mma<MTW, ROWS>(P0, Wo, ss + 5 * 64, true, nullptr, F0, lane, row0);
      res = F0;
    }
    team_sync();
    // ---- store [d][32] rows: lane = (row, chunk).  pad = 1 writes into a tensor with a replicated 1-voxel border
    //      ([D+2][H+2][W+2], what the trilinear-x2 "up2" GEMM consumes) ----
    const int ph = p / Wd, pw = p - ph * Wd;
    if (pad == 2) {
      // output [B][2D][H+2][W+2][32]: trilinear's depth axis is resolved here (x2, align_corners=False, clamped), the
      // h/w borders are replicated; the up2 GEMM (kind 2) then only interpolates bilinearly in (h, w)
      const int Dz = 2 * D, Hp2 = H + 2, Wp2 = Wd + 2;
      const size_t oplane = (size_t)B * Dz * Hp2 * Wp2 * AT_C;
      for (int z0 = 8 * wip; z0 < Dz; z0 += 8 * WPP) {
        const int z = z0 + (lane >> 2), q = lane & 3;
        if (z < Dz) {
          const int i = z >> 1;
          const int ia = (z & 1) ? i : max(i - 1, 0), ib = (z & 1) ? min(i + 1, D - 1) : i;
          const float wa = (z & 1) ? 0.75f : 0.25f, wb = 1.f - wa;
          float f[8];
          const float4 a0 = *reinterpret_cast<const float4*>(res + ia * AT_C + q * 8);
          const float4 a1 = *reinterpret_cast<const float4*>(res + ia * AT_C + q * 8 + 4);
          const float4 b0 = *reinterpret_cast<const float4*>(res + ib * AT_C + q * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(res + ib * AT_C + q * 8 + 4);
          f[0] = wa * a0.x + wb * b0.x; f[1] = wa * a0.y + wb * b0.y; f[2] = wa * a0.z + wb * b0.z; f[3] = wa * a0.w + wb * b0.w;
          f[4] = wa * a1.x + wb * b1.x; f[5] = wa * a1.y + wb * b1.y; f[6] = wa * a1.z + wb * b1.z; f[7] = wa * a1.w + wb * b1.w;
          for (int iy = 0; iy < 3; ++iy) {
            const int yy = iy == 0 ? ph + 1 : (iy == 1 ? (ph == 0 ? 0 : -1) : (ph == H - 1 ? H + 1 : -1));
            if (yy < 0) continue;
            for (int ix = 0; ix < 3; ++ix) {
              const int xx = ix == 0 ? pw + 1 : (ix == 1 ? (pw == 0 ? 0 : -1) : (pw == Wd - 1 ? Wd + 1 : -1));
              if (xx < 0) continue;
              store8<PLANES>(y, oplane, ((((size_t)b * Dz + z) * Hp2 + yy) * Wp2 + xx) * AT_C + q * 8, f);
            }
          }
        }
      }
      team_sync();
      continue;
    }
    const int Dp2 = D + 2 * pad, Hp2 = H + 2 * pad, Wp2 = Wd + 2 * pad;
    const size_t oplane = (size_t)B * Dp2 * Hp2 * Wp2 * AT_C;
    for (int d0 = 8 * wip; d0 < D; d0 += 8 * WPP) {
      const int d = d0 + (lane >> 2), q = lane & 3;
      if (d < D) {
        float f[8];
        const float4 a = *reinterpret_cast<const float4*>(res + d * AT_C + q * 8);
        const float4 c2 = *reinterpret_cast<const float4*>(res + d * AT_C + q * 8 + 4);
        f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = c2.x; f[5] = c2.y; f[6] = c2.z; f[7] = c2.w;
        if (!pad) {
          store8<PLANES>(y, oplane, (((size_t)b * D + d) * HW + p) * AT_C + q * 8, f);
        } else {
          // every coordinate x in [0,n) maps to x+1, plus the replicated border copies 0 (x==0) and n+1 (x==n-1)
          for (int iz = 0; iz < 3; ++iz) {
            const int zz = iz == 0 ? d + 1 : (iz == 1 ? (d == 0 ? 0 : -1) : (d == D - 1 ? D + 1 : -1));
            if (zz < 0) continue;
            for (int iy = 0; iy < 3; ++iy) {
              const int yy = iy == 0 ? ph + 1 : (iy == 1 ? (ph == 0 ? 0 : -1) : (ph == H - 1 ? H + 1 : -1));
              if (yy < 0) continue;
              for (int ix = 0; ix < 3; ++ix) {
                const int xx = ix == 0 ? pw + 1 : (ix == 1 ? (pw == 0 ? 0 : -1) : (pw == Wd - 1 ? Wd + 1 : -1));
                if (xx < 0) continue;
                store8<PLANES>(y, oplane, ((((size_t)b * Dp2 + zz) * Hp2 + yy) * Wp2 + xx) * AT_C + q * 8, f);
              }
            }
          }
        }
      }
    }
    team_sync();
  }
}

// ------------------------------------------------------------------------------------------------
// trilinear x2 (align_corners=False) of t [B,Dl,Hl,Wl,32] + Wc . cost [B,2Dl,2Hl,2Wl,32], then BN.
//   out[v] = scale * (up(t)[v] + Wc cost[v]) + shift
// A warp owns one 2x2x2 output block whose 8 voxels share the same 8 low-res corners
// (block index i in [-1, n-1] per axis -> outputs {2i+1, 2i+2} clipped to [0, 2n)).
// lane = (voxel v of the block, channel octet q): every global access is a 16-byte vector, the four
// lanes of a voxel cover its 64-byte channel row.  The 32x32 matvec reads the block's cost vectors
// (padded rows) and Wc from shared memory with conflict-free LDS.128.
// ------------------------------------------------------------------------------------------------
constexpr int UF_WARPS = 8;

struct UfBlock {            // raw prefetched data of one 2x2x2 block for this lane
  uint4 c_hi, c_lo;         // cost octet of the lane's voxel
  uint4 k_hi, k_lo;         // corner (lane>>2), octet (lane&3) of t
  size_t ooff;
  bool valid;
};

template <int PLANES>
__device__ __forceinline__ void uf_fetch(UfBlock& u, long long blk, const __nv_bfloat16* __restrict__ t,
                                         const __nv_bfloat16* __restrict__ cost, int Dl, int Hl, int Wl, int nbd,
                                         int nbh, int nbw, int lane, size_t lplane, size_t hplane) {
  const int D = 2 * Dl, H = 2 * Hl, W = 2 * Wl;
  long long r = blk;
  const int bw = (int)(r % nbw) - 1; r /= nbw;
  const int bh = (int)(r % nbh) - 1; r /= nbh;
  const int bd = (int)(r % nbd) - 1;
  const int b = (int)(r / nbd);
  const int v = lane >> 2, q = lane & 3;
  const int a = v >> 2, bb = (v >> 1) & 1, c = v & 1;
  const int oz = 2 * bd + 1 + a, oy = 2 * bh + 1 + bb, ox = 2 * bw + 1 + c;
  u.valid = oz >= 0 && oz < D && oy >= 0 && oy < H && ox >= 0 && ox < W;
  u.ooff = ((((size_t)b * D + (u.valid ? oz : 0)) * H + (u.valid ? oy : 0)) * W + (u.valid ? ox : 0)) * AT_C + q * 8;
  u.c_hi = u.c_lo = make_uint4(0, 0, 0, 0);
  if (u.valid) {
    u.c_hi = *reinterpret_cast<const uint4*>(cost + u.ooff);
    if (PLANES == 2) u.c_lo = *reinterpret_cast<const uint4*>(cost + hplane + u.ooff);
  }
  // corner (a,bb,c) of the block, clamped
  const int iz = min(max(bd + a, 0), Dl - 1), iy = min(max(bh + bb, 0), Hl - 1), ix = min(max(bw + c, 0), Wl - 1);
  const size_t koff = ((((size_t)b * Dl + iz) * Hl + iy) * Wl + ix) * AT_C + q * 8;
  u.k_hi = *reinterpret_cast<const uint4*>(t + koff);
  u.k_lo = make_uint4(0, 0, 0, 0);
  if (PLANES == 2) u.k_lo = *reinterpret_cast<const uint4*>(t + lplane + koff);
}

template <int PLANES>
__global__ void __launch_bounds__(UF_WARPS * 32, 2)
upsample_fuse_kernel(const __nv_bfloat16* __restrict__ t, const __nv_bfloat16* __restrict__ cost,
                     const float* __restrict__ WcT, const float* __restrict__ scale, const float* __restrict__ shift,
                     __nv_bfloat16* __restrict__ y, int B, int Dl, int Hl, int Wl) {
  __shared__ __align__(16) float ws[AT_C * AT_C];            // Wc transposed [ci][co]
  __shared__ __align__(16) float cs[UF_WARPS][8][AT_C + 4];  // cost vectors  [warp][voxel][channel] (padded rows)
  __shared__ __align__(16) float kn[UF_WARPS][8][AT_C + 4];  // corner vectors [warp][corner][channel]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int v = lane >> 2, q = lane & 3;
  for (int i = threadIdx.x; i < AT_C * AT_C; i += blockDim.x) ws[i] = __ldg(WcT + i);
  __shared__ __align__(16) float s_sc[AT_C], s_sh[AT_C];
  if (threadIdx.x < AT_C) { s_sc[threadIdx.x] = __ldg(scale + threadIdx.x); s_sh[threadIdx.x] = __ldg(shift + threadIdx.x); }
  __syncthreads();
  const size_t lplane = (size_t)B * Dl * Hl * Wl * AT_C, hplane = lplane * 8;
  const int nbd = Dl + 1, nbh = Hl + 1, nbw = Wl + 1;
  const long long nblocks = (long long)B * nbd * nbh * nbw;
  const int a = v >> 2, bb = (v >> 1) & 1, c = v & 1;
  // output 2i+1 (first of the pair): .75*in[i] + .25*in[i+1];  output 2i+2: .25*in[i] + .75*in[i+1]
  const float wz0 = a ? 0.25f : 0.75f, wy0 = bb ? 0.25f : 0.75f, wx0 = c ? 0.25f : 0.75f;
  const long long stride = (long long)gridDim.x * UF_WARPS;
  long long blk = (long long)blockIdx.x * UF_WARPS + warp;
  UfBlock cur;
  if (blk < nblocks) uf_fetch<PLANES>(cur, blk, t, cost, Dl, Hl, Wl, nbd, nbh, nbw, lane, lplane, hplane);
  for (; blk < nblocks; blk += stride) {
    UfBlock nxt;
    const bool has_next = blk + stride < nblocks;
    if (has_next) uf_fetch<PLANES>(nxt, blk + stride, t, cost, Dl, Hl, Wl, nbd, nbh, nbw, lane, lplane, hplane);
    // ---- stage this block: cost octet of voxel v, corner octet of corner v ----
    {
      float f[8], g[8];
      unpack8(cur.c_hi, f);
      if (PLANES == 2) { unpack8(cur.c_lo, g);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] += g[j]; }
      float4* crow = reinterpret_cast<float4*>(&cs[warp][v][q * 8]);
      crow[0] = make_float4(f[0], f[1], f[2], f[3]);
      crow[1] = make_float4(f[4], f[5], f[6], f[7]);
      unpack8(cur.k_hi, f);
      if (PLANES == 2) { unpack8(cur.k_lo, g);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] += g[j]; }
      float4* krow = reinterpret_cast<float4*>(&kn[warp][v][q * 8]);
      krow[0] = make_float4(f[0], f[1], f[2], f[3]);
      krow[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
    __syncwarp();
    // ---- trilinear blend of the 8 corners for this lane's voxel / octet ----
    float up[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) up[j] = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float wgt = ((k >> 2) ? 1.f - wz0 : wz0) * (((k >> 1) & 1) ? 1.f - wy0 : wy0) * ((k & 1) ? 1.f - wx0 : wx0);
      const float4 k0 = *reinterpret_cast<const float4*>(&kn[warp][k][q * 8]);
      const float4 k1 = *reinterpret_cast<const float4*>(&kn[warp][k][q * 8 + 4]);
      up[0] = fmaf(wgt, k0.x, up[0]); up[1] = fmaf(wgt, k0.y, up[1]); up[2] = fmaf(wgt, k0.z, up[2]);
      up[3] = fmaf(wgt, k0.w, up[3]); up[4] = fmaf(wgt, k1.x, up[4]); up[5] = fmaf(wgt, k1.y, up[5]);
      up[6] = fmaf(wgt, k1.z, up[6]); up[7] = fmaf(wgt, k1.w, up[7]);
    }
    // ---- 32x32 matvec: this lane's 8 output channels of its voxel ----
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
    for (int c4 = 0; c4 < AT_C; c4 += 4) {
      const float4 xv = *reinterpret_cast<const float4*>(&cs[warp][v][c4]);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float4 w0 = *reinterpret_cast<const float4*>(&ws[(c4 + u) * AT_C + q * 8]);
        const float4 w1 = *reinterpret_cast<const float4*>(&ws[(c4 + u) * AT_C + q * 8 + 4]);
        acc[0] = fmaf(xs[u], w0.x, acc[0]); acc[1] = fmaf(xs[u], w0.y, acc[1]);
        acc[2] = fmaf(xs[u], w0.z, acc[2]); acc[3] = fmaf(xs[u], w0.w, acc[3]);
        acc[4] = fmaf(xs[u], w1.x, acc[4]); acc[5] = fmaf(xs[u], w1.y, acc[5]);
        acc[6] = fmaf(xs[u], w1.z, acc[6]); acc[7] = fmaf(xs[u], w1.w, acc[7]);
      }
    }
    if (cur.valid) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (up[j] + acc[j]) * s_sc[q * 8 + j] + s_sh[q * 8 + j];
      store8<PLANES>(y, hplane, cur.ooff, o);
    }
    __syncwarp();
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------
// softmax over disparity fused with soft-argmin regression; the probability volume never exists.
// logits fp32 [B,D,H,W] -> pred [B,H,W].  thread = pixel.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
softmax_regress_kernel(const float* __restrict__ logits, float* __restrict__ pred, int D, int HW) {
  const int b = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float* lp = logits + (size_t)b * D * HW + p;
  float m = -INFINITY;
  for (int d = 0; d < D; ++d) m = fmaxf(m, lp[(size_t)d * HW]);
  float s = 0.f, acc = 0.f;
  for (int d = 0; d < D; ++d) {
    const float ev = expf(lp[(size_t)d * HW] - m);
    s += ev;
    acc = fmaf(ev, (float)d, acc);
  }
  pred[(size_t)b * HW + p] = acc / s;
}

// disparity_regression of the reference (submodule.py:127-131) on its own: pred = sum_d d * x[d], x = whatever the
// caller passes (probabilities in the reference's use; NOT renormalised here).  thread = pixel, fp32.
__global__ void __launch_bounds__(256)
regress_f32_kernel(const float* __restrict__ x, float* __restrict__ pred, int D, int HW) {
  const int b = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float* xp = x + (size_t)b * D * HW + p;
  float acc = 0.f;
  for (int d = 0; d < D; ++d) acc = fmaf(xp[(size_t)d * HW], (float)d, acc);
  pred[(size_t)b * HW + p] = acc;
}

// ------------------------------------------------------------------------------------------------
// convex 4x upsampling.  mask fp32 channels-last [B,H,W,144] (c = n*16 + i*4 + j), disp [B,H,W],
// out [B,1,4H,4W].  thread = (pixel, sub-row i): softmax over the 9 neighbours for its 4 columns.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
convex_upsample_kernel(const float* __restrict__ mask, const float* __restrict__ disp, float* __restrict__ out, int B,
                       int H, int W) {
  const size_t total = (size_t)B * H * W * 4;
  pdl_wait();
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx & 3);
    size_t pix = idx >> 2;
    const int w = (int)(pix % W);
    const int h = (int)((pix / W) % H);
    const int b = (int)(pix / ((size_t)W * H));
    const float* mp = mask + pix * 144 + i * 4;
    float4 mv[9];
    float dv[9];
#pragma unroll
    for (int n = 0; n < 9; ++n) {
      mv[n] = *reinterpret_cast<const float4*>(mp + n * 16);
      const int hh = h + n / 3 - 1, ww = w + n % 3 - 1;
      dv[n] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? 4.f * __ldg(disp + ((size_t)b * H + hh) * W + ww) : 0.f;
    }
    float4 mx = mv[0];
#pragma unroll
    for (int n = 1; n < 9; ++n) {
      mx.x = fmaxf(mx.x, mv[n].x); mx.y = fmaxf(mx.y, mv[n].y); mx.z = fmaxf(mx.z, mv[n].z); mx.w = fmaxf(mx.w, mv[n].w);
    }
    float4 s = make_float4(0, 0, 0, 0), a = make_float4(0, 0, 0, 0);
#pragma unroll
    for (int n = 0; n < 9; ++n) {
      const float ex = expf(mv[n].x - mx.x), ey = expf(mv[n].y - mx.y), ez = expf(mv[n].z - mx.z),
                  ew = expf(mv[n].w - mx.w);
      s.x += ex; s.y += ey; s.z += ez; s.w += ew;
      a.x = fmaf(ex, dv[n], a.x); a.y = fmaf(ey, dv[n], a.y); a.z = fmaf(ez, dv[n], a.z); a.w = fmaf(ew, dv[n], a.w);
    }
    float4 o = make_float4(a.x / s.x, a.y / s.y, a.z / s.z, a.w / s.w);
    *reinterpret_cast<float4*>(out + ((size_t)b * 4 * H + 4 * h + i) * (4 * W) + 4 * w) = o;
  }
}

// ------------------------------------------------------------------------------------------------
// softmax + disparity regression + convex 4x upsampling in ONE kernel (gwcnet_dca_g.py:238-239 + :117-124) for callers
// that hold the classif3 LOGITS: a CTA owns a 32 x 8 tile of 1/4-res pixels, regresses the disparity of the tile and its
// 1-pixel ring (recomputed by the neighbouring CTAs: 1.33x the 5.75 MB logits, instead of a grid-wide dependency)
// into shared memory (zero outside the image = F.unfold(padding=1)), writes the tile's own 1/4-res disparities, then
// upsamples from shared memory.  Same formulas as softmax_regress_kernel / convex_upsample_kernel: bit-identical.
// ------------------------------------------------------------------------------------------------
constexpr int RU_TW = 32, RU_TH = 8;
__global__ void __launch_bounds__(RU_TW * RU_TH)
softmax_regress_upsample_kernel(const float* __restrict__ logits, const float* __restrict__ mask, float* __restrict__ pred_q,
                                float* __restrict__ out, int B, int D, int H, int W) {
  __shared__ float s_d[RU_TH + 2][RU_TW + 2];
  const int b = blockIdx.z, h0 = blockIdx.y * RU_TH, w0 = blockIdx.x * RU_TW;
  const size_t HW = (size_t)H * W;
  pdl_wait();
  for (int i = threadIdx.x; i < (RU_TH + 2) * (RU_TW + 2); i += blockDim.x) {
    const int ly = i / (RU_TW + 2), lx = i - ly * (RU_TW + 2);
    const int h = h0 + ly - 1, w = w0 + lx - 1;
    float v = 0.f;
    if (h >= 0 && h < H && w >= 0 && w < W) {
      const float* lp = logits + (size_t)b * D * HW + (size_t)h * W + w;
      float m = -INFINITY;
      for (int d = 0; d < D; ++d) m = fmaxf(m, lp[(size_t)d * HW]);
      float sum = 0.f, acc = 0.f;
      for (int d = 0; d < D; ++d) {
        const float ev = expf(lp[(size_t)d * HW] - m);
        sum += ev;
        acc = fmaf(ev, (float)d, acc);
      }
      v = acc / sum;
      if (ly >= 1 && ly <= RU_TH && lx >= 1 && lx <= RU_TW) pred_q[(size_t)b * HW + (size_t)h * W + w] = v;
    }
    s_d[ly][lx] = v;
  }
  __syncthreads();
  for (int it = threadIdx.x; it < RU_TW * RU_TH * 4; it += blockDim.x) {
    const int i = it & 3, px = it >> 2;
    const int lx = px % RU_TW, ly = px / RU_TW;
    const int h = h0 + ly, w = w0 + lx;
    if (h >= H || w >= W) continue;
    const float* mp = mask + (((size_t)b * H + h) * W + w) * 144 + i * 4;
    float4 mv[9];
    float dv[9];
#pragma unroll
    for (int n = 0; n < 9; ++n) {
      mv[n] = *reinterpret_cast<const float4*>(mp + n * 16);
      dv[n] = 4.f * s_d[ly + n / 3][lx + n % 3];
    }
    float4 mx = mv[0];
#pragma unroll
    for (int n = 1; n < 9; ++n) {
      mx.x = fmaxf(mx.x, mv[n].x); mx.y = fmaxf(mx.y, mv[n].y); mx.z = fmaxf(mx.z, mv[n].z); mx.w = fmaxf(mx.w, mv[n].w);
    }
    float4 sm = make_float4(0, 0, 0, 0), a = make_float4(0, 0, 0, 0);
#pragma unroll
    for (int n = 0; n < 9; ++n) {
      const float ex = expf(mv[n].x - mx.x), ey = expf(mv[n].y - mx.y), ez = expf(mv[n].z - mx.z),
                  ew = expf(mv[n].w - mx.w);
      sm.x += ex; sm.y += ey; sm.z += ez; sm.w += ew;
      a.x = fmaf(ex, dv[n], a.x); a.y = fmaf(ey, dv[n], a.y); a.z = fmaf(ez, dv[n], a.z); a.w = fmaf(ew, dv[n], a.w);
    }
    *reinterpret_cast<float4*>(out + ((size_t)b * 4 * H + 4 * h + i) * (4 * W) + 4 * w) =
        make_float4(a.x / sm.x, a.y / sm.y, a.z / sm.z, a.w / sm.w);
  }
}

// ------------------------------------------------------------------------------------------------
// layout conversion between the reference's fp32 NCDHW tensors and cost planes
// ------------------------------------------------------------------------------------------------
template <int PLANES>
__global__ void __launch_bounds__(256)
planes_from_ncdhw_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int C, int Cp,
                         size_t V) {
  // V = D*H*W voxels per batch item; thread = (b, c8, voxel) with voxel fastest (coalesced reads)
  const int c8n = Cp / 8;
  const size_t total = (size_t)B * c8n * V;
  const size_t plane = (size_t)B * V * Cp;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t v = i % V;
    const int c8 = (int)((i / V) % c8n);
    const int b = (int)(i / (V * c8n));
    float f[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = c8 * 8 + k;
      f[k] = (c < C) ? __ldg(x + ((size_t)b * C + c) * V + v) : 0.f;
    }
    store8<PLANES>(y, plane, ((size_t)b * V + v) * Cp + c8 * 8, f);
  }
}

__global__ void __launch_bounds__(256)
planes_to_ncdhw_kernel(const __nv_bfloat16* __restrict__ x, int planes, float* __restrict__ y, int B, int C, int Cp,
                       size_t V, size_t ybs) {
  const size_t total = (size_t)B * C * V;
  const size_t plane = (size_t)B * V * Cp;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t v = i % V;
    const int c = (int)((i / V) % C);
    const int b = (int)(i / (V * C));
    const size_t off = ((size_t)b * V + v) * Cp + c;
    float r = h16_bits_to_float(__bfloat16_as_ushort(x[off]));
    if (planes == 2) r += h16_bits_to_float(__bfloat16_as_ushort(x[plane + off]));
    y[(size_t)b * ybs + (size_t)c * V + v] = r;
  }
}

// Tiled form for Cp % 8 == 0: a block transposes 64 voxels x Cp channels through shared memory, so that both the plane
// reads (16-byte vectors along the channel rows) and the NCHW writes (256-byte runs along the voxels) are coalesced
// (the element-per-thread form above reads with a stride of Cp elements: 65 us for 128 channels at 96x312x2).
constexpr int P2N_TV = 64;
__global__ void __launch_bounds__(256)
planes_to_nchw_tiled_kernel(const __nv_bfloat16* __restrict__ x, int planes, float* __restrict__ y, int B, int C, int Cp,
                            size_t V, size_t ybs) {
  extern __shared__ float p2n_tile[];                   // [Cp][P2N_TV + 1]
  const int b = blockIdx.y;
  const size_t v0 = (size_t)blockIdx.x * P2N_TV;
  const size_t plane = (size_t)B * V * Cp;
  const int c8n = Cp >> 3;
  for (int i = threadIdx.x; i < P2N_TV * c8n; i += blockDim.x) {
    const int vox = i / c8n, c8 = i - vox * c8n;
    if (v0 + vox >= V) continue;
    const size_t off = ((size_t)b * V + v0 + vox) * Cp + (size_t)c8 * 8;
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(x + off), f);
    if (planes == 2) {
      float g[8];
      unpack8(*reinterpret_cast<const uint4*>(x + plane + off), g);
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] += g[k];
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) p2n_tile[(c8 * 8 + k) * (P2N_TV + 1) + vox] = f[k];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C * P2N_TV; i += blockDim.x) {
    const int c = i / P2N_TV, vox = i - c * P2N_TV;
    if (v0 + vox < V) y[(size_t)b * ybs + (size_t)c * V + v0 + vox] = p2n_tile[c * (P2N_TV + 1) + vox];
  }
}

static int launch_planes_to_nchw(const void* x, int planes, float* y, int B, int C, int Cp, size_t V, size_t ybs,
                                 cudaStream_t st) {
  const size_t total = (size_t)B * C * V;
  const size_t smem = (size_t)Cp * (P2N_TV + 1) * sizeof(float);
  if ((Cp % 8) == 0 && smem <= 48 * 1024 && B <= 65535 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    dim3 grid((unsigned)((V + P2N_TV - 1) / P2N_TV), (unsigned)B);
    planes_to_nchw_tiled_kernel<<<grid, 256, smem, st>>>((const __nv_bfloat16*)x, planes, y, B, C, Cp, V, ybs);
  } else {
    const size_t nb = (total + 255) / 256;
    const size_t cap = (size_t)dca_num_sms() * 16;
    planes_to_ncdhw_kernel<<<(unsigned)(nb < cap ? (nb ? nb : 1) : cap), 256, 0, st>>>((const __nv_bfloat16*)x, planes, y, B, C, Cp, V, ybs);
  }
  return 0;
}

// weights: torch Conv [Co][Ci][taps] or ConvTranspose [Ci][Co][taps] -> [taps][Ci][CoPad] fp32 (zero pad)
__global__ void pack_weight_kernel(const float* __restrict__ w, int transposed, int Co, int Ci, int taps,
                                   float* __restrict__ out, int CoPad) {
  const int total = taps * Ci * CoPad;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int co = i % CoPad, ci = (i / CoPad) % Ci, t = i / (CoPad * Ci);
    float v = 0.f;
    if (co < Co) v = transposed ? w[((size_t)ci * Co + co) * taps + t] : w[((size_t)co * Ci + ci) * taps + t];
    out[i] = v;
  }
}

// eval-mode BatchNorm -> per-channel scale/shift (length Cpad, identity padding)
__global__ void fold_bn_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                               const float* __restrict__ mean, const float* __restrict__ var, float eps,
                               float* __restrict__ scale, float* __restrict__ shift, int C, int Cpad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cpad) return;
  if (i < C) {
    const float s = gamma[i] / sqrtf(var[i] + eps);
    scale[i] = s;
    shift[i] = beta[i] - mean[i] * s;
  } else {
    scale[i] = 1.f; shift[i] = 0.f;
  }
}

// out[b,d,h,w] = sum over the 27 taps (kd,kh,kw) of P[tap][b, d+kd-1, h+kh-1, w+kw-1] (zero outside): the shifted
// sum that turns the per-tap products of dca_conv1_taps_tc into the 3x3x3 conv to one channel.  P is tap-major, so
// every one of a thread's 27 loads is coalesced along w.
__global__ void __launch_bounds__(256)
tap_gather3d_kernel(const float* __restrict__ P, float* __restrict__ out, int B, int D, int H, int W) {
  const size_t nvox = (size_t)B * D * H * W;
  const int HW = H * W;
  pdl_wait();
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvox; v += (size_t)gridDim.x * blockDim.x) {
    const int w = (int)(v % W);
    size_t r = v / W;
    const int h = (int)(r % H); r /= H;
    const int d = (int)(r % D);
    // unconditional, independent loads (an out-of-volume tap reads the centre voxel and is multiplied by 0)
    float val[27];
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
      const bool okd = (d + kd - 1 >= 0) && (d + kd - 1 < D);
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const bool okh = okd && (h + kh - 1 >= 0) && (h + kh - 1 < H);
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const bool ok = okh && (w + kw - 1 >= 0) && (w + kw - 1 < W);
          const long long nb = ok ? ((long long)(kd - 1) * HW + (kh - 1) * W + (kw - 1)) : 0ll;
          val[(kd * 3 + kh) * 3 + kw] = __ldg(P + (size_t)((kd * 3 + kh) * 3 + kw) * nvox + v + nb) * (ok ? 1.f : 0.f);
        }
      }
    }
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < 27; ++t) acc += val[t];
    out[v] = acc;
  }
}

// Fused tail of classif3 (gwcnet_dca_g.py:235-239): logit[d] = 27-tap shifted sum of P (as tap_gather3d), then
// softmax over d and disparity regression -- the logits and the probability volume never reach HBM.
// Block = 32 w-columns x DG disparity groups of one image row; a thread walks its disparity chunk with an online
// softmax (running max / sum / weighted sum), the DG partial states of a pixel are merged through shared memory.
// Every load is coalesced along w.  logits_out (optional): the summed logits [B,D,H,W] (stage-count variants with no
// cva stage return them).
template <int TG_DG>
__global__ void __launch_bounds__(32 * TG_DG)
tap_gather_softmax_regress_kernel(const float* __restrict__ P, float* __restrict__ pred, float* __restrict__ logits_out,
                                  int B, int D, int H, int W) {
  __shared__ float s_m[TG_DG][32], s_s[TG_DG][32], s_a[TG_DG][32];
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int w = blockIdx.x * 32 + lane, h = blockIdx.y, b = blockIdx.z;
  const size_t nvox = (size_t)B * D * H * W;
  const int chunk = (D + TG_DG - 1) / TG_DG;
  const int d0 = g * chunk, d1 = min(D, d0 + chunk);
  float m = -INFINITY, sum = 0.f, acc = 0.f;
  pdl_wait();
  if (w < W) {
    // in-plane validity of the 9 (kh, kw) neighbours and their clamped offsets (an invalid tap reads the centre voxel,
    // its value is discarded): the 27 loads of a voxel are UNCONDITIONAL and independent, so they are all in flight
    // together (a branch per tap serialised one DRAM latency per load)
    float ok9[9];
    int off9[9];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const bool ok = (h + kh - 1 >= 0) && (h + kh - 1 < H) && (w + kw - 1 >= 0) && (w + kw - 1 < W);
        ok9[kh * 3 + kw] = ok ? 1.f : 0.f;
        off9[kh * 3 + kw] = ok ? (kh - 1) * W + (kw - 1) : 0;
      }
    const int HW = H * W;
    for (int d = d0; d < d1; ++d) {
      const size_t v = (((size_t)b * D + d) * H + h) * W + w;
      float val[27];
#pragma unroll
      for (int kd = 0; kd < 3; ++kd) {
        const bool okd = (d + kd - 1 >= 0) && (d + kd - 1 < D);
        const float* base = P + (size_t)(kd * 9) * nvox + v + (okd ? (long long)(kd - 1) * HW : 0ll);
#pragma unroll
        for (int t = 0; t < 9; ++t) val[kd * 9 + t] = __ldg(base + (size_t)t * nvox + off9[t]) * (okd ? ok9[t] : 0.f);
      }
      float logit = 0.f;
#pragma unroll
      for (int t = 0; t < 27; ++t) logit += val[t];
      if (logits_out) logits_out[v] = logit;
      const float mn = fmaxf(m, logit);
      const float corr = expf(m - mn), ev = expf(logit - mn);      // first step: exp(-inf) = 0
      sum = sum * corr + ev;
      acc = acc * corr + ev * (float)d;
      m = mn;
    }
  }
  s_m[g][lane] = m; s_s[g][lane] = sum; s_a[g][lane] = acc;
  __syncthreads();
  if (g == 0 && w < W) {
    float M = s_m[0][lane];
#pragma unroll
    for (int i = 1; i < TG_DG; ++i) M = fmaxf(M, s_m[i][lane]);
    float S = 0.f, A = 0.f;
#pragma unroll
    for (int i = 0; i < TG_DG; ++i) {
      const float sc = (s_s[i][lane] > 0.f) ? expf(s_m[i][lane] - M) : 0.f;     // empty chunks carry m = -inf, s = 0
      S = fmaf(s_s[i][lane], sc, S);
      A = fmaf(s_a[i][lane], sc, A);
    }
    pred[((size_t)b * H + h) * W + w] = A / S;
  }
}

// ------------------------------------------------------------------------------------------------
// The two 3-channel stems of the front end: Conv2d(3 -> 32, K x K, stride 2, pad K/2) (+ bias) + BN + ReLU --
// feature_extraction.firstconv[0] (3x3, gwcnet_dca_g.py:19) and Guidance.conv_start (7x7, submodule.py:413-414).
// Too few input channels for the tensor-core family and only 0.2 / 0.6 GMAC: thread = output pixel with all 32 output
// channels in registers, weights transposed to [tap][ci][co] in shared memory (every lane reads the same address:
// broadcast float4 loads), fp32 NCHW image in, cost planes [P][B][1][Ho][Wo][32] out (no layout pass in between).
// ------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(128)
conv2d_stem_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ scale,
                   const float* __restrict__ shift, __nv_bfloat16* __restrict__ y, int planes, int B, int H, int W, int Ho,
                   int Wo, int act) {
  __shared__ __align__(16) float sw[K * K * 3 * 32];
  __shared__ float ssc[32], ssh[32];
  for (int i = threadIdx.x; i < K * K * 3 * 32; i += blockDim.x) {
    const int co = i & 31, t = i >> 5, ci = t % 3, kk = t / 3;
    sw[i] = w[(co * 3 + ci) * K * K + kk];
  }
  if (threadIdx.x < 32) {
    ssc[threadIdx.x] = scale ? scale[threadIdx.x] : 1.f;
    ssh[threadIdx.x] = shift ? shift[threadIdx.x] : 0.f;
  }
  __syncthreads();
  const size_t npix = (size_t)B * Ho * Wo;
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= npix) return;
  const int ox = (int)(pix % Wo), oy = (int)((pix / Wo) % Ho), b = (int)(pix / ((size_t)Wo * Ho));
  float acc[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) acc[c] = 0.f;
  const float* xb = x + (size_t)b * 3 * H * W;
  for (int kh = 0; kh < K; ++kh) {
    const int iy = 2 * oy + kh - K / 2;
    if (iy < 0 || iy >= H) continue;
    for (int kw = 0; kw < K; ++kw) {
      const int ix = 2 * ox + kw - K / 2;
      if (ix < 0 || ix >= W) continue;
      const float* wp = sw + (kh * K + kw) * 3 * 32;
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        const float v = __ldg(xb + ((size_t)ci * H + iy) * W + ix);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 ww = *reinterpret_cast<const float4*>(wp + ci * 32 + 4 * c4);
          acc[4 * c4 + 0] = fmaf(v, ww.x, acc[4 * c4 + 0]); acc[4 * c4 + 1] = fmaf(v, ww.y, acc[4 * c4 + 1]);
          acc[4 * c4 + 2] = fmaf(v, ww.z, acc[4 * c4 + 2]); acc[4 * c4 + 3] = fmaf(v, ww.w, acc[4 * c4 + 3]);
        }
      }
    }
  }
  const size_t plane = npix * 32;
#pragma unroll
  for (int c8 = 0; c8 < 4; ++c8) {
    float o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = apply_act(fmaf(acc[8 * c8 + k], ssc[8 * c8 + k], ssh[8 * c8 + k]), act);
    store8_rt(y, plane, planes, pix * 32 + 8 * c8, o);
  }
}

static inline int grid_for(size_t total, int threads) {
  size_t g = (total + threads - 1) / threads;
  const size_t cap = (size_t)dca_num_sms() * 32;
  return (int)(g < cap ? (g ? g : 1) : cap);
}

}  // namespace dca

using namespace dca;

// thread-per-output form (any C % 8 == 0); dca_avgpool3d (conv_tc.cu) takes the TMA-staged depth-marching kernel for C == 32
extern "C" int dca_avgpool3d_simple(const void* x, void* y, int planes, int B, int C, int Di, int Hi, int Wi, void* stream) {
  if (!x || !y || C % 8 != 0 || B <= 0 || Di <= 0 || Hi <= 0 || Wi <= 0 || planes < 1 || planes > 2)
    return DCA_ERR_ARG;
  const int Do = (Di + 1) / 2, Ho = (Hi + 1) / 2, Wo = (Wi + 1) / 2;
  const size_t total = (size_t)B * Do * Ho * Wo * (C / 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (planes == 2)
    avgpool3d_kernel<2><<<grid_for(total, 256), 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, B, C, Di, Hi,
                                                               Wi, Do, Ho, Wo);
  else
    avgpool3d_kernel<1><<<grid_for(total, 256), 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, B, C, Di, Hi,
                                                               Wi, Do, Ho, Wo);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_class_stats(const float* logits, int* cls, float* e, float* S, void* scratch, int B, int D, int H,
                               int W, void* stream) {
  // scratch: (B*D + 1) x 8 bytes, 8-byte aligned (fixed-point sums + ticket); zeroed here
  if (!logits || !cls || !e || !S || !scratch || ((uintptr_t)scratch & 7) || B <= 0 || D <= 0 || D > CS_MAXD || H <= 0 ||
      W <= 0)
    return DCA_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(scratch, 0, ((size_t)B * D + 1) * sizeof(unsigned long long), st) != cudaSuccess) return DCA_ERR_LAUNCH;
  const int HW = H * W;
  dca_launch(class_stats_kernel, dim3((HW + 31) / 32, B), CS_THREADS, 0, st, logits, cls, e, S,
             (unsigned long long*)scratch, D, HW, B * D);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

static int g_attention_team = 1;
// D/8 == 24: 1 (default) = two warps per pixel + mma.sync attention core, 2 = two warps + fp32 FMA core, 0 = one warp
extern "C" int dca_attention_set_team(int on) { g_attention_team = on; return DCA_OK; }

static int attention_launch(const void* x, const int* cls, const float* e, const float* S, const float* weights,
                            int has_wa, void* y, int pad, int planes, int B, int C, int D, int H, int W,
                            const void* key, void* stream) {
  if (pad < 0 || pad > 2) return DCA_ERR_ARG;
  if (!x || (!key && (!cls || !e || !S)) || !weights || !y || planes < 1 || planes > 2 || B <= 0 || D <= 0) return DCA_ERR_ARG;
  if (C != AT_C) return DCA_ERR_UNSUPPORTED;
  const int MT = (D + 15) / 16;
  if (MT > 4) return DCA_ERR_UNSUPPORTED;
  const size_t wbytes = (size_t)AT_NMAT * 2 * AT_WPLANE * 2 + 6 * 64 * 4;
  const bool core = (D == 24 && g_attention_team == 1);          // tensor-core attention core: 4 hi/lo pair buffers per team
  const size_t pair_bytes = (size_t)(2 * 16 * MT * AT_PITCH) * 2;
  const size_t per_warp = core ? 4 * pair_bytes : 2 * pair_bytes + (size_t)3 * (16 * MT * AT_C) * 4;   // per pixel in flight
  int warps = core ? 9 : 8;
  while (warps > 1 && wbytes + warps * per_warp > 224 * 1024) --warps;
  const size_t smem = wbytes + warps * per_warp;
  const int HW = H * W;
  int grid = (B * HW + warps - 1) / warps;
  if (grid > dca_num_sms()) grid = dca_num_sms();            // persistent: one CTA per SM pays the weight-staging prologue once
  cudaStream_t st = (cudaStream_t)stream;
#define DCA_AT_LAUNCH2(P_, MT_, DT_, WPP_, CORE_)                                                                      \
  do {                                                                                                           \
    auto kern = disp_attention_kernel<P_, MT_, DT_, WPP_, CORE_>;                                                          \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                          \
    dca_launch(kern, grid, warps * 32 * WPP_, smem, st, (const __nv_bfloat16*)x, cls, e, S, weights, has_wa,       \
               (__nv_bfloat16*)y, B, D, H, W, pad, (const __nv_bfloat16*)key);                                    \
  } while (0)
#define DCA_AT_LAUNCH(P_, MT_) DCA_AT_LAUNCH2(P_, MT_, 0, 1, 0)
  if (D == 24 && g_attention_team == 1) {          // two warps per pixel, tensor-core attention core
    if (planes == 2) DCA_AT_LAUNCH2(2, 2, 24, 2, 1); else DCA_AT_LAUNCH2(1, 2, 24, 2, 1);
  } else if (D == 24 && g_attention_team == 2) {   // two warps per pixel, fp32 FMA core
    if (planes == 2) DCA_AT_LAUNCH2(2, 2, 24, 2, 0); else DCA_AT_LAUNCH2(1, 2, 24, 2, 0);
  } else if (D == 24) {
    if (planes == 2) DCA_AT_LAUNCH2(2, 2, 24, 1, 0); else DCA_AT_LAUNCH2(1, 2, 24, 1, 0);
  } else if (planes == 2) {
    if (MT == 1) DCA_AT_LAUNCH(2, 1); else if (MT == 2) DCA_AT_LAUNCH(2, 2); else if (MT == 3) DCA_AT_LAUNCH(2, 3); else DCA_AT_LAUNCH(2, 4);
  } else {
    if (MT == 1) DCA_AT_LAUNCH(1, 1); else if (MT == 2) DCA_AT_LAUNCH(1, 2); else if (MT == 3) DCA_AT_LAUNCH(1, 3); else DCA_AT_LAUNCH(1, 4);
  }
#undef DCA_AT_LAUNCH
#undef DCA_AT_LAUNCH2
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_disp_attention(const void* x, const int* cls, const float* e, const float* S, const float* weights,
                                  int has_wa, void* y, int pad, int planes, int B, int C, int D, int H, int W,
                                  void* stream) {
  return attention_launch(x, cls, e, S, weights, has_wa, y, pad, planes, B, C, D, H, W, nullptr, stream);
}

// SelfAttentionBlock.forward(query_feats, key_feats) (SelfAttention_bn.py:62-98), the generic two-input form:
// q = Pq1(Pq0(query)), k = Pk1(Pk0(key)), v = Pv(key), out = Po(softmax(q k^T / sqrt(8)) v) per pixel over the D axis.
// query, key, y: cost planes [P][B][D][H][W][32]; weights as for dca_disp_attention (the 7th matrix is unused).
extern "C" int dca_self_attention(const void* query, const void* key, const float* weights, void* y, int planes, int B,
                                  int C, int D, int H, int W, void* stream) {
  if (!key) return DCA_ERR_ARG;
  return attention_launch(query, nullptr, nullptr, nullptr, weights, 0, y, 0, planes, B, C, D, H, W, key, stream);
}

extern "C" int dca_upsample_fuse(const void* t, const void* cost, const float* WcT, const float* scale,
                                 const float* shift, void* y, int planes, int B, int C, int Dl, int Hl, int Wl,
                                 void* stream) {
  if (!t || !cost || !WcT || !scale || !shift || !y || planes < 1 || planes > 2 || B <= 0) return DCA_ERR_ARG;
  if (C != AT_C) return DCA_ERR_UNSUPPORTED;
  const long long nblocks = (long long)B * (Dl + 1) * (Hl + 1) * (Wl + 1);
  const size_t gcap = (size_t)dca_num_sms() * 12;
  int grid = (int)((nblocks + 7) / 8 < gcap ? (nblocks + 7) / 8 : gcap);
  cudaStream_t st = (cudaStream_t)stream;
  if (planes == 2)
    upsample_fuse_kernel<2><<<grid, 256, 0, st>>>((const __nv_bfloat16*)t, (const __nv_bfloat16*)cost, WcT, scale,
                                                  shift, (__nv_bfloat16*)y, B, Dl, Hl, Wl);
  else
    upsample_fuse_kernel<1><<<grid, 256, 0, st>>>((const __nv_bfloat16*)t, (const __nv_bfloat16*)cost, WcT, scale,
                                                  shift, (__nv_bfloat16*)y, B, Dl, Hl, Wl);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_softmax_regress(const float* logits, float* pred, int B, int D, int H, int W, void* stream) {
  if (!logits || !pred || B <= 0 || D <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  const int HW = H * W;
  softmax_regress_kernel<<<dim3((HW + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(logits, pred, D, HW);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

// logits fp32 [B,D,H,W], mask fp32 channels-last [B,H,W,144] -> pred_q [B,1,H,W] (1/4-res disparity) and out [B,1,4H,4W],
// one launch (softmax_regress_upsample_kernel).
extern "C" int dca_softmax_regress_upsample(const float* logits, const float* mask, float* pred_q, float* out, int B, int D,
                                            int H, int W, void* stream) {
  if (!logits || !mask || !pred_q || !out || B <= 0 || D <= 0 || H <= 0 || W <= 0 || B > 65535) return DCA_ERR_ARG;
  dca_launch(softmax_regress_upsample_kernel, dim3((W + RU_TW - 1) / RU_TW, (H + RU_TH - 1) / RU_TH, B), RU_TW * RU_TH, 0,
             (cudaStream_t)stream, logits, mask, pred_q, out, B, D, H, W);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_regress_f32(const float* x, float* pred, int B, int D, int H, int W, void* stream) {
  if (!x || !pred || B <= 0 || D <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  const int HW = H * W;
  regress_f32_kernel<<<dim3((HW + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(x, pred, D, HW);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_convex_upsample(const float* mask, const float* disp, float* out, int B, int H, int W,
                                   void* stream) {
  if (!mask || !disp || !out || B <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  const size_t total = (size_t)B * H * W * 4;
  dca_launch(convex_upsample_kernel, grid_for(total, 256), 256, 0, (cudaStream_t)stream, mask, disp, out, B, H, W);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_tap_gather3d(const float* P, float* out, int B, int D, int H, int W, void* stream) {
  if (!P || !out || B <= 0 || D <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  const size_t total = (size_t)B * D * H * W;
  dca_launch(tap_gather3d_kernel, grid_for(total, 256), 256, 0, (cudaStream_t)stream, P, out, B, D, H, W);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

static int g_tg_dg = 16;
extern "C" int dca_tap_gather_set_groups(int n) { g_tg_dg = n; return DCA_OK; }
// P fp32 tap-major [27][B*D*H*W] (dca_conv3d_tc_taps27 / dca_conv1_taps_tc) -> pred [B,H,W] = sum_d d softmax_d(logits),
// logits = 27-tap shifted sum of P; logits_out optional ([B,D,H,W]).  Replaces tap_gather3d + softmax_regress.
extern "C" int dca_tap_gather_softmax_regress(const float* P, float* pred, float* logits_out, int B, int D, int H, int W,
                                              void* stream) {
  if (!P || !pred || B <= 0 || D <= 0 || H <= 0 || W <= 0 || H > 65535 || B > 65535) return DCA_ERR_ARG;
  // disparity groups per block (threads = 32 x groups; each thread walks D / groups disparities with 27 loads in flight).
  // Measured at KITTI (benchmarks/one_tail.py): 4: 43.5 us, 6: 69.8, 8: 55.4, 16: 39.7 (default; 155 MB -> 3.9 TB/s = 0.60 of
  // measured HBM), 24 / 32: 76.8 -- the stride pattern of the 27 x D plane reads, not the thread count, decides
  const dim3 grid((W + 31) / 32, H, B);
  cudaStream_t st = (cudaStream_t)stream;
  switch (g_tg_dg) {
    case 8: dca_launch(tap_gather_softmax_regress_kernel<8>, grid, 32 * 8, 0, st, P, pred, logits_out, B, D, H, W); break;
    case 4: dca_launch(tap_gather_softmax_regress_kernel<4>, grid, 32 * 4, 0, st, P, pred, logits_out, B, D, H, W); break;
    case 6: dca_launch(tap_gather_softmax_regress_kernel<6>, grid, 32 * 6, 0, st, P, pred, logits_out, B, D, H, W); break;
    case 24: dca_launch(tap_gather_softmax_regress_kernel<24>, grid, 32 * 24, 0, st, P, pred, logits_out, B, D, H, W); break;
    case 32: dca_launch(tap_gather_softmax_regress_kernel<32>, grid, 32 * 32, 0, st, P, pred, logits_out, B, D, H, W); break;
    default: dca_launch(tap_gather_softmax_regress_kernel<16>, grid, 32 * 16, 0, st, P, pred, logits_out, B, D, H, W); break;
  }
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_planes_from_ncdhw(const float* x, void* y, int planes, int B, int C, int Cp, int D, int H, int W,
                                     void* stream) {
  if (!x || !y || planes < 1 || planes > 2 || B <= 0 || C <= 0 || Cp < C || Cp % 8 != 0) return DCA_ERR_ARG;
  const size_t V = (size_t)D * H * W, total = (size_t)B * (Cp / 8) * V;
  cudaStream_t st = (cudaStream_t)stream;
  if (planes == 2)
    planes_from_ncdhw_kernel<2><<<grid_for(total, 256), 256, 0, st>>>(x, (__nv_bfloat16*)y, B, C, Cp, V);
  else
    planes_from_ncdhw_kernel<1><<<grid_for(total, 256), 256, 0, st>>>(x, (__nv_bfloat16*)y, B, C, Cp, V);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_planes_to_ncdhw(const void* x, int planes, float* y, int B, int C, int Cp, int D, int H, int W,
                                   void* stream) {
  if (!x || !y || planes < 1 || planes > 2 || B <= 0 || C <= 0 || Cp < C) return DCA_ERR_ARG;
  const size_t V = (size_t)D * H * W;
  launch_planes_to_nchw(x, planes, y, B, C, Cp, V, (size_t)C * V, (cudaStream_t)stream);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

// Same, into a CHANNEL SLICE of a wider fp32 NCHW tensor: y points at the slice's first channel of batch 0 and
// y_batch_stride (elements) is the batch pitch of the wide tensor -- how feature_extraction's torch.cat((l2, l3, l4))
// (gwcnet_dca_g.py:60) is written without a copy.
extern "C" int dca_planes_to_nchw_slice(const void* x, int planes, float* y, int B, int C, int Cp, int H, int W,
                                        long long y_batch_stride, void* stream) {
  if (!x || !y || planes < 1 || planes > 2 || B <= 0 || C <= 0 || Cp < C || y_batch_stride < (long long)C * H * W)
    return DCA_ERR_ARG;
  launch_planes_to_nchw(x, planes, y, B, C, Cp, (size_t)H * W, (size_t)y_batch_stride, (cudaStream_t)stream);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_pack_weights(const float* w, int transposed, int Co, int Ci, int taps, float* out, int CoPad,
                                void* stream) {
  if (!w || !out || Co <= 0 || Ci <= 0 || taps <= 0 || CoPad < Co) return DCA_ERR_ARG;
  pack_weight_kernel<<<grid_for((size_t)taps * Ci * CoPad, 256), 256, 0, (cudaStream_t)stream>>>(w, transposed, Co, Ci,
                                                                                                 taps, out, CoPad);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_fold_bn(const float* gamma, const float* beta, const float* mean, const float* var, float eps,
                           float* scale, float* shift, int C, int Cpad, void* stream) {
  if (!gamma || !beta || !mean || !var || !scale || !shift || C <= 0 || Cpad < C) return DCA_ERR_ARG;
  fold_bn_kernel<<<(Cpad + 127) / 128, 128, 0, (cudaStream_t)stream>>>(gamma, beta, mean, var, eps, scale, shift, C,
                                                                       Cpad);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_conv2d_stem(const float* x, const float* w, const float* scale, const float* shift, void* y, int planes,
                               int act, int B, int H, int W, int K, void* stream) {
  if (!x || !w || !y || planes < 1 || planes > 2 || B <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  if (K != 3 && K != 7) return DCA_ERR_UNSUPPORTED;
  const int Ho = (H + 2 * (K / 2) - K) / 2 + 1, Wo = (W + 2 * (K / 2) - K) / 2 + 1;
  const size_t npix = (size_t)B * Ho * Wo;
  const unsigned grid = (unsigned)((npix + 127) / 128);
  cudaStream_t st = (cudaStream_t)stream;
  if (K == 3)
    conv2d_stem_kernel<3><<<grid, 128, 0, st>>>(x, w, scale, shift, (__nv_bfloat16*)y, planes, B, H, W, Ho, Wo, act);
  else
    conv2d_stem_kernel<7><<<grid, 128, 0, st>>>(x, w, scale, shift, (__nv_bfloat16*)y, planes, B, H, W, Ho, Wo, act);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

// F.adaptive_avg_pool3d of the rows [h0, H) of an fp32 [B][D][H][W] tensor to [B][Do][Ho][Wo] (torch's windows:
// [floor(i*In/Out), ceil((i+1)*In/Out)) per axis) -- the visualisation head of the plain-GwcNet baseline,
// models/gwcnet.py:186-190.  thread = output element.
__global__ void __launch_bounds__(256)
adaptive_avgpool3d_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int D, int H, int W, int h0, int Do,
                          int Ho, int Wo) {
  const size_t total = (size_t)B * Do * Ho * Wo;
  const int Hi = H - h0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ow = (int)(i % Wo), oh = (int)((i / Wo) % Ho), od = (int)((i / ((size_t)Wo * Ho)) % Do);
    const int b = (int)(i / ((size_t)Wo * Ho * Do));
    const int d0 = (int)(((long long)od * D) / Do), d1 = (int)(((long long)(od + 1) * D + Do - 1) / Do);
    const int a0 = (int)(((long long)oh * Hi) / Ho), a1 = (int)(((long long)(oh + 1) * Hi + Ho - 1) / Ho);
    const int w0 = (int)(((long long)ow * W) / Wo), w1 = (int)(((long long)(ow + 1) * W + Wo - 1) / Wo);
    float s = 0.f;
    for (int d = d0; d < d1; ++d)
      for (int h = a0; h < a1; ++h)
        for (int w = w0; w < w1; ++w) s += x[(((size_t)b * D + d) * H + h0 + h) * W + w];
    y[i] = s / (float)((d1 - d0) * (a1 - a0) * (w1 - w0));
  }
}

extern "C" int dca_adaptive_avgpool3d_rows(const float* x, float* y, int B, int D, int H, int W, int h0, int Do, int Ho,
                                           int Wo, void* stream) {
  if (!x || !y || B <= 0 || D <= 0 || H <= 0 || W <= 0 || h0 < 0 || h0 >= H || Do <= 0 || Ho <= 0 || Wo <= 0) return DCA_ERR_ARG;
  const size_t total = (size_t)B * Do * Ho * Wo;
  adaptive_avgpool3d_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, y, B, D, H, W, h0, Do, Ho, Wo);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

static int g_pdl = 1;
extern "C" int dca_pdl_enabled(void) { return g_pdl; }
// 1 (default): kernels are launched with programmatic stream serialization (PDL, dca_common.cuh); 0: fully serialised
extern "C" int dca_set_pdl(int on) { g_pdl = on ? 1 : 0; return DCA_OK; }

extern "C" int dca_version(void) { return 102; }
// 16-bit format of the cost planes and operand packs this build was compiled for: 1 = IEEE fp16 (default), 0 = bf16
extern "C" int dca_plane_format(void) { return DCA_F16_PLANES ? 1 : 0; }
