// Fused group-wise-correlation + concat cost volume (SURVEY 8a rows a1+a2).
// Replaces the reference's two Python loops over disparities
//   build_gwc_volume     /root/reference/models/submodule.py:157-167 (groupwise_correlation :148-154)
//   build_concat_volume  /root/reference/models/submodule.py:134-145
// and the torch.cat at models/gwcnet_dca_g.py:220.
//
// HBM-bound: reads 2 x (C + Cc) x H x W fp32 once (re-reads of the right-image window hit L2),
// writes [B][D][H][W][Cv] bf16 (x planes) once with sector-complete stores.
//
// Fused kernel layout
//   CTA  = one (b, h) row, TW=16 columns, one chunk of DC<=48 disparities; 256 threads.
//   smem = left tile  Ls[c][w][g]  (c = channel inside its group, g = group, pitch G+1)
//          right tile Rs[c][u][g]  for the u = w-d window (zero-filled outside the image)
//          concat tiles (channel-major).
//   warp = 4 columns x 8 disparities, lane = output channel slot (0..31 then 32..63):
//          slot < G  -> group correlation (register tile 4w x 8d: 15 LDS per 32 FMA)
//          G <= slot < G+Cc -> left concat copy, < G+2Cc -> right concat copy, rest zero pad.
//   The 32 fp32 results of a lane are bf16-split, pair-exchanged by shuffle and stored as 32-bit
//   words so that a warp store covers whole 32-byte sectors of two voxels.
#include <cuda.h>

#include "dca_common.cuh"

namespace dca {

constexpr int VOL_TW = 16;   // columns per CTA
constexpr int VOL_DC = 48;   // disparities per CTA
constexpr int VOL_THREADS = 256;

// 4-byte async global->shared copy (LDGSTS); src_size 0 zero-fills the destination (out-of-image columns)
__device__ __forceinline__ void cp_async4(float* dst, const float* src, bool valid) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src),
               "r"(valid ? 4 : 0)
               : "memory");
}

__device__ __forceinline__ void vol_split2(float a, float b, uint32_t& hi, uint32_t& lo) { split_pair(a, b, hi, lo); }

// LiDAR guidance of the guided instantiations (include/dca_b200.h section 14): every channel of volume plane d at a
// 1/4-res pixel with hq > 0 is multiplied by k * expf(-(t * t) * s), t = d - hq, before the hi/lo split.  The unguided
// instantiations never read it.
struct VolGuide { const float* hq; float k, s; };
__device__ __forceinline__ float guide_factor(const VolGuide& g, float hv, int d) {
  const float t = (float)d - hv;
  return g.k * expf(-(t * t) * g.s);
}

// CVT = compile-time channel pitch of the volume (64 for DCANet's 40 groups + 2x12 concat); 0 = runtime Cv.
// GT / CPGT = compile-time group count / channels per group (40 / 8 for DCANet); 0 = runtime.  With them fixed
// every shared-memory offset of the inner product loop is an immediate and the channel loop unrolls fully.
// GUIDED: lane (j, i) = (lane / 4, lane % 4) of a warp tile computes the factor of (d0+dt+j, w0+wt+i) once; the store
// fetches it by shuffle.
template <int PLANES, int CVT, int GT, int CPGT, bool GUIDED = false>
__global__ void __launch_bounds__(VOL_THREADS, 2)
volume_fused_kernel(const float* __restrict__ gl, const float* __restrict__ gr,
                    const float* __restrict__ cl, const float* __restrict__ cr,
                    __nv_bfloat16* __restrict__ vol, int B, int C, int G_rt, int Cc, int D, int H, int W, int Cv_rt,
                    const VolGuide guide) {
  extern __shared__ float smem[];
  const int Cv = CVT ? CVT : Cv_rt;
  const int G = GT ? GT : G_rt;
  const int cpg = CPGT ? CPGT : C / G;
  const int gp = G + 1;                       // pitch of the group axis (bank-conflict-free transposing stores)
  constexpr int UW = VOL_TW + VOL_DC - 1;     // right window width (63)
  float* Ls = smem;                           // [cpg][TW][gp]
  float* Rs = Ls + cpg * VOL_TW * gp;         // [cpg][UW][gp]
  float* cLs = Rs + cpg * UW * gp;            // [Cc][TW]
  float* cRs = cLs + Cc * VOL_TW;             // [Cc][UW]

  const int wtiles = (W + VOL_TW - 1) / VOL_TW;
  const int w0 = (blockIdx.x % wtiles) * VOL_TW;
  const int dchunk = blockIdx.x / wtiles;
  const int d0 = dchunk * VOL_DC;
  const int h = blockIdx.y, b = blockIdx.z;
  const int dcount = min(VOL_DC, D - d0);
  const int u0 = w0 - (d0 + VOL_DC - 1);      // image column of window index 0
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const size_t HW = (size_t)H * W;

  // ---- stage: coalesced along w in global, transposed into [c][w][g] in smem (no div/mod in the loops) ----
  {
    // all copies are asynchronous (no register round trip): every thread has ~100 loads in flight at once
    const float* src = gl + ((size_t)b * C * H + h) * W;   // + ch*HW + w
    for (int i = tid; i < C * VOL_TW; i += VOL_THREADS) {
      const int ch = i / VOL_TW, wl = i % VOL_TW, w = w0 + wl;
      const bool ok = w < W;
      cp_async4(&Ls[((ch % cpg) * VOL_TW + wl) * gp + ch / cpg], ok ? src + (size_t)ch * HW + w : src, ok);
    }
    const float* srcr = gr + ((size_t)b * C * H + h) * W;
    for (int i = tid; i < C * UW; i += VOL_THREADS) {
      const int ch = i / UW, ul = i % UW, u = u0 + ul;
      const bool ok = u >= 0 && u < W;
      cp_async4(&Rs[((ch % cpg) * UW + ul) * gp + ch / cpg], ok ? srcr + (size_t)ch * HW + u : srcr, ok);
    }
    if (Cc > 0) {
      const float* s2 = cl + ((size_t)b * Cc * H + h) * W;
      for (int i = tid; i < Cc * VOL_TW; i += VOL_THREADS) {
        const int ch = i / VOL_TW, wl2 = i % VOL_TW, w = w0 + wl2;
        const bool ok = w < W;
        cp_async4(&cLs[i], ok ? s2 + (size_t)ch * HW + w : s2, ok);
      }
      const float* s3 = cr + ((size_t)b * Cc * H + h) * W;
      for (int i = tid; i < Cc * UW; i += VOL_THREADS) {
        const int ch = i / UW, ul = i % UW, u = u0 + ul;
        const bool ok = u >= 0 && u < W;
        cp_async4(&cRs[i], ok ? s3 + (size_t)ch * HW + u : s3, ok);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  }
  __syncthreads();

  const float inv_cpg = 1.0f / (float)cpg;
  const size_t plane_stride = (size_t)B * D * H * W * Cv;
  const int n_wt = VOL_TW / 4, n_dt = (dcount + 7) / 8;
  const int odd = lane & 1;

  for (int t = warp; t < n_wt * n_dt; t += VOL_THREADS / 32) {
    const int wt = (t % n_wt) * 4;            // local column of the 4-wide tile
    const int dt = (t / n_wt) * 8;            // local disparity of the 8-deep tile
    // window index of (w = w0+wt+i, d = d0+dt+j):  ul = wt + i - dt - j + (VOL_DC-1)
    const int ubase = wt - dt + (VOL_DC - 1) - 7;   // ul = ubase + (i - j + 7), i-j+7 in [0,10]
    float gf = 1.f;
    if (GUIDED) {
      const int w = w0 + wt + (lane & 3);
      const float hv = w < W ? guide.hq[((size_t)b * H + h) * W + w] : 0.f;
      if (hv > 0.f) gf = guide_factor(guide, hv, d0 + dt + (lane >> 2));
    }
    for (int pass = 0; pass < 2; ++pass) {
      const int slot = lane + 32 * pass;
      if (32 * pass >= Cv) break;
      float acc[8][4];
#pragma unroll
      for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;

      if (slot < G) {
#pragma unroll
        for (int c = 0; c < (CPGT ? CPGT : cpg); ++c) {
          float l[4], r[11];
          const float* lp = Ls + (c * VOL_TW + wt) * gp + slot;
          const float* rp = Rs + (c * UW + ubase) * gp + slot;
#pragma unroll
          for (int i = 0; i < 4; ++i) l[i] = lp[i * gp];
#pragma unroll
          for (int k = 0; k < 11; ++k) r[k] = rp[k * gp];
#pragma unroll
          for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[j][i] = fmaf(l[i], r[i - j + 7], acc[j][i]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[j][i] *= inv_cpg;
      } else if (slot < G + Cc) {
        const int cc = slot - G;
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i)
            acc[j][i] = (w0 + wt + i >= d0 + dt + j) ? cLs[cc * VOL_TW + wt + i] : 0.f;
      } else if (slot < G + 2 * Cc) {
        const int cc = slot - G - Cc;
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[j][i] = cRs[cc * UW + ubase + (i - j + 7)];
      }
      // ---- pair exchange (even lane keeps column ip, odd lane column ip+1), packed bf16 split, 32-bit stores ----
      const int ch = slot & ~1;
      const bool ch_ok = ch < Cv;
      // this lane's column inside each pair is ip + odd
      __nv_bfloat16* colp = vol + ((((size_t)b * D + d0 + dt) * H + h) * W + (w0 + wt + odd)) * Cv + ch;
      const size_t dstep = HW * Cv;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool d_ok = (dt + j) < dcount;
#pragma unroll
        for (int ip = 0; ip < 4; ip += 2) {
          const float mine_a = acc[j][ip], mine_b = acc[j][ip + 1];
          const float got = __shfl_xor_sync(0xffffffffu, odd ? mine_a : mine_b, 1);
          // even lane: voxel a, channels (slot, slot+1) = (mine_a, got); odd lane: voxel b, (slot-1, slot) = (got, mine_b)
          float lo_ch = odd ? got : mine_a, hi_ch = odd ? mine_b : got;
          if (GUIDED) {
            const float f = __shfl_sync(0xffffffffu, gf, j * 4 + ip + odd);
            lo_ch *= f;
            hi_ch *= f;
          }
          if (d_ok && ch_ok && (w0 + wt + ip + odd) < W) {
            uint32_t hw, lw;
            vol_split2(lo_ch, hi_ch, hw, lw);
            __nv_bfloat16* dst = colp + (size_t)j * dstep + ip * Cv;
            *reinterpret_cast<uint32_t*>(dst) = hw;
            if (PLANES == 2) *reinterpret_cast<uint32_t*>(dst + plane_stride) = lw;
          }
        }
      }
    }
  }
}

// =====================================================================================================
// TMA-staged fused kernel for DCANet's shape (C = 320 = 40 groups x 8, 12 concat channels, W % 8 == 0).
//   lane < G/2 owns the group PAIR (2l, 2l+1) = output channels (2l, 2l+1); a 4w x 8d register tile per group costs
//   4 LDS.128 per 32 FMA, and the two results of a voxel are exactly one packed bf16x2 word per plane: no shuffles, a
//   warp store = one voxel's 128-byte channel row.  Lanes G/2 .. G/2+Cc-1 copy the left / right concat features in the
//   same product form (cl[w] * [w >= d], 1 * cr[w-d]), the rest write the zero pad.
//   The window of a (row, 16 columns, 48 disparities) item starts at u0 = w0 - d0 - 48 (a multiple of 16 columns), is
//   64 columns wide and out-of-image columns are zero filled by TMA (= the reference's zero-initialised volume).
// =====================================================================================================
constexpr int V2_TW = 16, V2_DC = 48, V2_UW = 64;    // columns / disparities per item, right window (incl. 1 spare column)

__device__ __forceinline__ void vol_split2b(float a, float b, uint32_t& hi, uint32_t& lo) { split_pair(a, b, hi, lo); }

// Persistent CTAs (one per SM, 12 warps), TMA-staged and double buffered:
//   * the transposition to [c][u/8][slot][8] is done by the TMA unit: the fp32 NCHW feature map is described as a 5-D
//     tensor (8 columns | group/2 (+ batch) | group parity | column octet | (channel-in-group, row)), so ONE box per
//     channel-in-group lands as 32-byte units [u/8][slot] with slot = (g & 1) * G/2 + g/2; out-of-image octets are zero
//     filled.  No LSU work, no registers, no address arithmetic for staging.  SWIZZLE_32B swaps the two float4 of a
//     unit in every other 128-byte row, which is exactly what makes a warp's float4 loads (lane stride 32 B) conflict
//     free; with G % 8 == 0 the swap bit of a lane is (slot >> 2) & 1, a per-lane constant.
//   * warps walk ONE continuous stream of 4w x 8d tiles (24 slots per item, slot s -> warp s % 12: two tiles per warp
//     and item, measured 3 % faster than 16 warps); an item's buffer is refilled (next-but-one item) by whichever warp finishes its
//     last tile (shared-memory counter), and announced through an mbarrier with expect_tx.
constexpr int V3_WARPS = 12, V3_THREADS = 32 * V3_WARPS;
constexpr int V3_SLOTS = (V2_TW / 4) * (V2_DC / 8);      // tile slots per item (24)

struct VolMaps { CUtensorMap r, l, cr, cl; };

__device__ __forceinline__ uint32_t v_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void v_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(v_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void v_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(v_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void v_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  const uint32_t addr = v_smem_u32(bar);
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void v_tma_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                         int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(v_smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(v_smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void v_tma_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(v_smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(v_smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

template <int G, int CPG, int CC>
struct Vol3Cfg {
  static constexpr int HG = G / 2, LW4 = V2_TW / 4, UW4 = V2_UW / 4, LW8 = V2_TW / 8, UW8 = V2_UW / 8;
  static constexpr int RQ = CPG * UW4 * G, LQ = CPG * LW4 * G;       // float4 counts (dense slot pitch G)
  static constexpr int R_BYTES = RQ * 16, L_BYTES = LQ * 16, CR_BYTES = CC * V2_UW * 4, CL_BYTES = CC * V2_TW * 4;
  static constexpr int BUF_BYTES = R_BYTES + L_BYTES + CR_BYTES + CL_BYTES;
  static constexpr int SMEM_BYTES = 2 * BUF_BYTES + 128 + 1024;      // + barriers/counters + alignment slack
  static constexpr int GUIDE_BYTES = V3_WARPS * 32 * 4;              // guided: one factor per (j, i) of a warp's tile
};

// KS (1, 2 or 4) lanes share one group pair, each summing CPG / KS of its channels (xor-butterfly at the end).  8 groups
// (40 channels each) run with KS = 4: 4 x 4 + 12 = 28 busy lanes instead of 16, 328 -> 191 us at KITTI size.  20 groups
// stay at KS = 1 (measured: KS = 2 is 8 % SLOWER, 152 vs 141 us -- the kernel is bound by its 32-bit store instructions,
// one 2 x CV-byte row per warp instruction, not by the lanes' FMA work).
// GUIDED: lane (j, i) = (lane / 4, lane % 4) computes the factor of (d0+dt+j, w0+wt+i) into its warp's 32 floats after
// the barriers; hq = 0 stores factor 1, and v * 1 = v.
template <int PLANES, int G, int CPG, int CC, int CV, int KS = 1, bool GUIDED = false>
__global__ void __launch_bounds__(V3_THREADS, 1)
volume_fused3_kernel(const __grid_constant__ VolMaps maps, __nv_bfloat16* __restrict__ vol, int B, int D, int H, int W,
                     int dbg, const VolGuide guide) {
  using Cfg = Vol3Cfg<G, CPG, CC>;
  constexpr int HG = Cfg::HG, LW4 = Cfg::LW4, UW4 = Cfg::UW4, LW8 = Cfg::LW8, UW8 = Cfg::UW8;
  constexpr int HGK = HG * KS, CPK = CPG / KS;      // lanes doing correlation work, channels per such lane
  static_assert((KS == 1 || KS == 2 || KS == 4) && CPG % KS == 0 && HGK + CC <= 32, "lane plan");
  static_assert(G % 4 == 0, "a 128-byte smem row holds 4 slots: the swap bit is ((slot >> 2) + octet * G / 4) & 1");
  extern __shared__ __align__(1024) uint8_t smem_v3[];
  uint8_t* base = smem_v3;                 // (kept a shared-space pointer: no generic loads in the inner loop)
  if (threadIdx.x == 0 && (v_smem_u32(base) & 255u) != 0) __trap();            // SWIZZLE_32B pattern repeats every 256 bytes
  uint64_t* full = reinterpret_cast<uint64_t*>(base + 2 * Cfg::BUF_BYTES);     // [2]
  unsigned* cnt = reinterpret_cast<unsigned*>(full + 2);                       // [2]

  const int wtiles = (W + V2_TW - 1) / V2_TW, dchunks = (D + V2_DC - 1) / V2_DC;
  const int per_row = wtiles * dchunks;
  const int n_items = per_row * H * B;
  const int my_items = (n_items > (int)blockIdx.x) ? (n_items - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const size_t HW = (size_t)H * W;

  auto issue = [&](int k) {
    const int item = (int)blockIdx.x + k * (int)gridDim.x, buf = k & 1;
    const int rowi = item / per_row, inrow = item - rowi * per_row;
    const int b = rowi / H, h = rowi - b * H;
    const int w0 = (inrow % wtiles) * V2_TW, d0 = (inrow / wtiles) * V2_DC;
    const int u0 = w0 - d0 - V2_DC;
    uint8_t* bb = base + buf * Cfg::BUF_BYTES;
    v_mbar_expect_tx(&full[buf], Cfg::BUF_BYTES);
    for (int c = 0; c < CPG; ++c) {
      v_tma_5d(bb + c * (UW8 * G * 32), &maps.r, &full[buf], 0, HG * b, 0, u0 >> 3, c * H + h);
      v_tma_5d(bb + Cfg::R_BYTES + c * (LW8 * G * 32), &maps.l, &full[buf], 0, HG * b, 0, w0 >> 3, c * H + h);
    }
    if (CC > 0) {
      v_tma_3d(bb + Cfg::R_BYTES + Cfg::L_BYTES, &maps.cr, &full[buf], u0, CC * b, h);
      v_tma_3d(bb + Cfg::R_BYTES + Cfg::L_BYTES + Cfg::CR_BYTES, &maps.cl, &full[buf], w0, CC * b, h);
    }
  };

  pdl_trigger();      // persistent single-wave grid (dca_common.cuh)
  pdl_wait();         // the feature maps come from the previous kernel / copy of the stream
  if (tid == 0) {
    v_mbar_init(&full[0], 1); v_mbar_init(&full[1], 1);
    cnt[0] = 0; cnt[1] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (my_items > 0) issue(0);
    if (my_items > 1) issue(1);
  }
  __syncthreads();

  const float lane_scale = lane < HGK ? 1.0f / (float)CPG : 1.0f;
  const int gl = lane < HGK ? lane / KS : lane - HGK + HG;     // "virtual lane": owner of output channels (2 gl, 2 gl + 1)
  const int ks = lane < HGK ? lane % KS : 0;
  const size_t plane_stride = (size_t)B * D * H * W * CV;
  for (int s = warp; s < my_items * V3_SLOTS; s += V3_WARPS) {
    const int k = s / V3_SLOTS, t = s - k * V3_SLOTS;
    const int item = (int)blockIdx.x + k * (int)gridDim.x, buf = k & 1;
    const int rowi = item / per_row, inrow = item - rowi * per_row;
    const int b = rowi / H, h = rowi - b * H;
    const int w0 = (inrow % wtiles) * V2_TW, d0 = (inrow / wtiles) * V2_DC;
    const int dcount = min(V2_DC, D - d0);
    const int u0 = w0 - d0 - V2_DC;                     // image column of window index 0 (multiple of 4)
    const int wq = t % LW4, wt = wq * 4;                // local column of the 4-wide tile
    const int dt = (t / LW4) * 8;                       // local disparity of the 8-deep tile
    const float4* Rq = reinterpret_cast<const float4*>(base + buf * Cfg::BUF_BYTES);     // [CPG][UW4][G]
    const float4* Lq = Rq + Cfg::RQ;                                                     // [CPG][LW4][G]
    const float4* cRq = Lq + Cfg::LQ;                                                    // [CC][UW4]
    const float4* cLq = cRq + CC * UW4;                                                  // [CC][LW4]
    v_mbar_wait(&full[buf], (uint32_t)((k >> 1) & 1));
    if (w0 + wt < W && dt < dcount && !(dbg & 1)) {
      // window index of (w0+wt+i, d0+dt+j) = wt + i - dt - j + 48 = ub + (i - j + 8),  ub = wt - dt + 40 (multiple of 4)
      const int ub = wt - dt + V2_DC - 8;
      float acc[2][8][4];
      if (lane < HGK) {
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
          for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[q][j][i] = 0.f;
        // unit (o, slot) = 32 bytes at ((c*W8 + o)*G + slot)*32; float4 `half` of it sits at 16*(half ^ swap(slot))
        const uint8_t* Rb = reinterpret_cast<const uint8_t*>(Rq);
        const uint8_t* Lb = reinterpret_cast<const uint8_t*>(Lq);
        const int ub4 = ub >> 2;
        uint32_t lo_[2], ro_[2][3];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          // SWIZZLE_32B swaps the two float4 of a unit in odd 128-byte rows; row = unit / 4 = (octet * G + slot) / 4, so
          // with G % 8 == 0 the bit is a per-lane constant and with G % 8 == 4 (20 groups) it flips with the octet
          const int slot = gl + q * HG, sw = (slot >> 2) & 1;
          constexpr int OSW = (G >> 2) & 1;
          lo_[q] = (uint32_t)((((wq >> 1) * G + slot) << 5) + (((wq & 1) ^ sw ^ (OSW & (wq >> 1))) << 4));
#pragma unroll
          for (int kk = 0; kk < 3; ++kk)
            ro_[q][kk] = (uint32_t)(((((ub4 + kk) >> 1) * G + slot) << 5) +
                                    ((((ub4 + kk) & 1) ^ sw ^ (OSW & ((ub4 + kk) >> 1))) << 4));
        }
#pragma unroll
        for (int cc_ = 0; cc_ < CPK; ++cc_) {
          const int c = ks * CPK + cc_;
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const float4 l4 = *reinterpret_cast<const float4*>(Lb + c * (LW8 * G * 32) + lo_[q]);
            const float4 r0 = *reinterpret_cast<const float4*>(Rb + c * (UW8 * G * 32) + ro_[q][0]),
                         r1 = *reinterpret_cast<const float4*>(Rb + c * (UW8 * G * 32) + ro_[q][1]),
                         r2 = *reinterpret_cast<const float4*>(Rb + c * (UW8 * G * 32) + ro_[q][2]);
            const float l[4] = {l4.x, l4.y, l4.z, l4.w};
            const float r[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
              for (int i = 0; i < 4; ++i) acc[q][j][i] = fmaf(l[i], r[i - j + 8], acc[q][j][i]);
          }
        }
        if (KS > 1) {                                   // sum the KS partial channel sums of a group pair
          constexpr unsigned m = HGK == 32 ? 0xffffffffu : ((1u << HGK) - 1u);
#pragma unroll
          for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                float v = acc[q][j][i];
                v += __shfl_xor_sync(m, v, 1);
                if (KS == 4) v += __shfl_xor_sync(m, v, 2);
                acc[q][j][i] = v;
              }
        }
      } else {
        // concat lanes, same product form: left copy = cl[w] * [w - d >= 0], right copy = 1 * cr[w - d]
        const bool left = lane < HGK + CC / 2;
        const int cc = 2 * (lane - HGK - (left ? 0 : CC / 2));
        const bool live = lane < HGK + CC;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float l[4] = {1.f, 1.f, 1.f, 1.f}, r[12];
          if (left) {
            const float4 l4 = live ? cLq[(cc + q) * LW4 + wq] : make_float4(0.f, 0.f, 0.f, 0.f);
            l[0] = l4.x; l[1] = l4.y; l[2] = l4.z; l[3] = l4.w;
#pragma unroll
            for (int kk = 0; kk < 12; ++kk) r[kk] = (u0 + ub + kk >= 0) ? 1.f : 0.f;
          } else {
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            const float4* rp = cRq + (cc + q) * UW4 + (ub >> 2);
            const float4 r0 = live ? rp[0] : z4, r1 = live ? rp[1] : z4, r2 = live ? rp[2] : z4;
            r[0] = r0.x; r[1] = r0.y; r[2] = r0.z; r[3] = r0.w; r[4] = r1.x; r[5] = r1.y; r[6] = r1.z; r[7] = r1.w;
            r[8] = r2.x; r[9] = r2.y; r[10] = r2.z; r[11] = r2.w;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[q][j][i] = l[i] * r[i - j + 8];
        }
      }
      float* gfw = reinterpret_cast<float*>(base + 2 * Cfg::BUF_BYTES + 128) + warp * 32;
      if (GUIDED) {
        const float hv = guide.hq[((size_t)b * H + h) * W + w0 + wt + (lane & 3)];     // W % 8 == 0: in the row
        gfw[lane] = hv > 0.f ? guide_factor(guide, hv, d0 + dt + (lane >> 2)) : 1.f;
        __syncwarp();
      }
      if (2 * gl < CV && ks == 0) {
        __nv_bfloat16* rowp = vol + ((((size_t)b * D + d0 + dt) * H + h) * W + (w0 + wt)) * CV + 2 * gl;
        // the 32 lanes own 2 * NVL channels; zero-pad channels beyond that (KS > 1 uses lanes up) fall to the last lane
        constexpr int NVL = 32 - HGK + HG;
        constexpr int NPAD = CV > 2 * NVL ? (CV - 2 * NVL) / 2 : 0;
        const bool pads = NPAD > 0 && gl == NVL - 1;
        const size_t dstep = HW * CV;
        const int nj = min(8, dcount - dt);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (j < nj) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint32_t hw, lw;
              if (GUIDED) {
                const float f = gfw[j * 4 + i];
                vol_split2b(acc[0][j][i] * lane_scale * f, acc[1][j][i] * lane_scale * f, hw, lw);
              } else {
                vol_split2b(acc[0][j][i] * lane_scale, acc[1][j][i] * lane_scale, hw, lw);
              }
              *reinterpret_cast<uint32_t*>(rowp + i * CV) = hw;
              if (PLANES == 2) *reinterpret_cast<uint32_t*>(rowp + plane_stride + i * CV) = lw;
              if (pads) {
#pragma unroll
                for (int z = 1; z <= NPAD; ++z) {
                  *reinterpret_cast<uint32_t*>(rowp + i * CV + 2 * z) = 0u;
                  if (PLANES == 2) *reinterpret_cast<uint32_t*>(rowp + plane_stride + i * CV + 2 * z) = 0u;
                }
              }
            }
          }
          rowp += dstep;
        }
      }
    }
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      const unsigned old = atomicAdd(&cnt[buf], 1u);
      if (old == V3_SLOTS - 1) {                        // last tile of this item: the buffer is free, refill it
        __threadfence_block();
        cnt[buf] = 0;
        if (k + 2 < my_items && !(dbg & 2)) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          issue(k + 2);
        } else if (k + 2 < my_items) {
          v_mbar_expect_tx(&full[buf], 0);              // (timing probe: no loads)
        }
      }
    }
  }
}

typedef CUresult (*VolEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static VolEncodeFn vol_get_encode() {
  static VolEncodeFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<VolEncodeFn>(sym);
  }
  return fn;
}

// features [B][G*CPG][H][W] fp32 as (8 | G/2 (+ batch) | 2 | W/8 | CPG*H), box = (8, G/2, 2, octets, 1), SWIZZLE_32B
static bool vol_feature_map(CUtensorMap* m, const float* p, int B, int G, int CPG, int H, int W, int octets) {
  VolEncodeFn enc = vol_get_encode();
  if (!enc) return false;
  const cuuint64_t HW = (cuuint64_t)H * W;
  cuuint64_t dims[5] = {8, (cuuint64_t)(G / 2) * B, 2, (cuuint64_t)(W / 8), (cuuint64_t)CPG * H};
  cuuint64_t strides[4] = {2 * (cuuint64_t)CPG * HW * 4, (cuuint64_t)CPG * HW * 4, 32, (cuuint64_t)W * 4};
  cuuint32_t box[5] = {8, (cuuint32_t)(G / 2), 2, (cuuint32_t)octets, 1};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(p), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// concat features [B][CC][H][W] fp32 as (W | CC*B | H), box = (cols, CC, 1)
static bool vol_concat_map(CUtensorMap* m, const float* p, int B, int CC, int H, int W, int cols) {
  VolEncodeFn enc = vol_get_encode();
  if (!enc) return false;
  const cuuint64_t HW = (cuuint64_t)H * W;
  cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)CC * B, (cuuint64_t)H};
  cuuint64_t strides[2] = {HW * 4, (cuuint64_t)W * 4};
  cuuint32_t box[3] = {(cuuint32_t)cols, (cuuint32_t)CC, 1};
  cuuint32_t es[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(p), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int g_vol_sms = 0;
static int g_volume_v2 = 1;   // bit0: use the TMA-staged kernel; bits 1..2: timing probes (skip compute / skip staging)
template <int G, int CPG, int CC, int CV, int KS, bool GUIDED>
static int launch_volume3(const float* gl, const float* gr, const float* cl, const float* cr, void* vol, int B, int D,
                          int H, int W, int planes, cudaStream_t st, const VolGuide& guide) {
  using Cfg = Vol3Cfg<G, CPG, CC>;
  static_assert(G % 2 == 0 && (G / 2) * KS + CC <= 32 && CV >= G + 2 * CC && CV <= 64 && Cfg::SMEM_BYTES <= 227 * 1024 &&
                Cfg::R_BYTES % 128 == 0 && Cfg::L_BYTES % 128 == 0 && Cfg::CR_BYTES % 128 == 0 && Cfg::CL_BYTES % 128 == 0,
                "shape");
  g_vol_sms = dca_num_sms();
  VolMaps maps;
  if (!vol_feature_map(&maps.r, gr, B, G, CPG, H, W, V2_UW / 8) || !vol_feature_map(&maps.l, gl, B, G, CPG, H, W, V2_TW / 8) ||
      !vol_concat_map(&maps.cr, cr, B, CC, H, W, V2_UW) || !vol_concat_map(&maps.cl, cl, B, CC, H, W, V2_TW))
    return DCA_ERR_LAUNCH;
  const int wtiles = (W + V2_TW - 1) / V2_TW, dchunks = (D + V2_DC - 1) / V2_DC;
  const long long items = (long long)wtiles * dchunks * H * B;
  if (items * V3_SLOTS >= (1ll << 31)) return DCA_ERR_UNSUPPORTED;
  const int grid = (int)(items < g_vol_sms ? items : g_vol_sms);
  const int smem = Cfg::SMEM_BYTES + (GUIDED ? Cfg::GUIDE_BYTES : 0);
  static_assert(Cfg::SMEM_BYTES + Cfg::GUIDE_BYTES <= 227 * 1024, "guided shared memory");
  if (planes == 2) {
    auto kern = volume_fused3_kernel<2, G, CPG, CC, CV, KS, GUIDED>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    dca_launch(kern, grid, V3_THREADS, smem, st, maps, (__nv_bfloat16*)vol, B, D, H, W, g_volume_v2 >> 1, guide);
  } else {
    auto kern = volume_fused3_kernel<1, G, CPG, CC, CV, KS, GUIDED>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    dca_launch(kern, grid, V3_THREADS, smem, st, maps, (__nv_bfloat16*)vol, B, D, H, W, g_volume_v2 >> 1, guide);
  }
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

// ---------------------------------------------------------------------------------------------
// Reference-API variants: fp32 NCDHW outputs, exactly the tensors build_gwc_volume /
// build_concat_volume return.  CTA = one (b, group, h) row staged in smem, lane = column,
// every thread walks the disparities; stores are coalesced along w.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gwc_volume_ncdhw_kernel(const float* __restrict__ gl, const float* __restrict__ gr, float* __restrict__ vol,
                        int B, int C, int G, int D, int H, int W) {
  extern __shared__ float smem[];
  const int cpg = C / G;
  float* Ls = smem;            // [cpg][W]
  float* Rs = smem + cpg * W;  // [cpg][W]
  const int h = blockIdx.x, g = blockIdx.y, b = blockIdx.z;
  const size_t HW = (size_t)H * W;
  const float* lsrc = gl + ((size_t)(b * C + g * cpg) * H + h) * W;
  const float* rsrc = gr + ((size_t)(b * C + g * cpg) * H + h) * W;
  for (int i = threadIdx.x; i < cpg * W; i += blockDim.x) {
    int c = i / W, w = i % W;
    Ls[i] = __ldg(lsrc + (size_t)c * HW + w);
    Rs[i] = __ldg(rsrc + (size_t)c * HW + w);
  }
  __syncthreads();
  const float inv = 1.0f / (float)cpg;
  for (int i = threadIdx.x; i < D * W; i += blockDim.x) {
    int d = i / W, w = i % W;
    float acc = 0.f;
    if (w >= d) {
      for (int c = 0; c < cpg; ++c) acc = fmaf(Ls[c * W + w], Rs[c * W + w - d], acc);
      acc *= inv;
    }
    vol[((((size_t)b * G + g) * D + d) * H + h) * W + w] = acc;
  }
}

__global__ void __launch_bounds__(256)
concat_volume_ncdhw_kernel(const float* __restrict__ cl, const float* __restrict__ cr, float* __restrict__ vol,
                           int B, int C, int D, int H, int W) {
  // one thread per output element of the [B,2C,D,H,W] volume, w fastest
  const size_t total = (size_t)B * 2 * C * D * H * W;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int w = (int)(i % W);
    size_t r = i / W;
    int h = (int)(r % H); r /= H;
    int d = (int)(r % D); r /= D;
    int c2 = (int)(r % (2 * C));
    int b = (int)(r / (2 * C));
    float v = 0.f;
    if (w >= d) {
      if (c2 < C) v = __ldg(cl + (((size_t)b * C + c2) * H + h) * W + w);
      else v = __ldg(cr + (((size_t)b * C + (c2 - C)) * H + h) * W + w - d);
    }
    vol[i] = v;
  }
}

}  // namespace dca

using namespace dca;

// 1 (default) = 16-byte-staged pair kernel for the DCANet shapes, 0 = generic kernel everywhere (A/B timing, tests)
extern "C" int dca_volume_set_v2(int on) { g_volume_v2 = on; return DCA_OK; }

namespace dca {
template <bool GUIDED>
static int volume_gwc_concat(const float* gwc_l, const float* gwc_r, const float* cat_l, const float* cat_r, void* vol,
                             int B, int C, int G, int Cc, int D, int H, int W, int Cv, int planes, void* stream,
                             const VolGuide& guide) {
  if (!gwc_l || !gwc_r || !vol || B <= 0 || C <= 0 || G <= 0 || D <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  if (C % G != 0 || (Cc > 0 && (!cat_l || !cat_r)) || Cc < 0) return DCA_ERR_ARG;
  if (Cv < G + 2 * Cc || Cv > 64 || (Cv % 8) != 0 || (planes != 1 && planes != 2)) return DCA_ERR_ARG;
  const int cpg = C / G, gp = G + 1, UW = VOL_TW + VOL_DC - 1;
  cudaStream_t st = (cudaStream_t)stream;
  if ((W % 8) == 0 && Cc == 12 && C == 320 && (g_volume_v2 & 1)) {      // DCANet's shape (40 groups) and the 20- and 8-group points of config 4's sweep
    if (G == 40 && Cv == 64) return launch_volume3<40, 8, 12, 64, 1, GUIDED>(gwc_l, gwc_r, cat_l, cat_r, vol, B, D, H, W, planes, st, guide);
    if (G == 20 && Cv == 64) return launch_volume3<20, 16, 12, 64, 1, GUIDED>(gwc_l, gwc_r, cat_l, cat_r, vol, B, D, H, W, planes, st, guide);
    if (G == 20 && Cv == 48) return launch_volume3<20, 16, 12, 48, 1, GUIDED>(gwc_l, gwc_r, cat_l, cat_r, vol, B, D, H, W, planes, st, guide);
    if (G == 8 && Cv == 32) return launch_volume3<8, 40, 12, 32, 4, GUIDED>(gwc_l, gwc_r, cat_l, cat_r, vol, B, D, H, W, planes, st, guide);
    if (G == 8 && Cv == 64) return launch_volume3<8, 40, 12, 64, 4, GUIDED>(gwc_l, gwc_r, cat_l, cat_r, vol, B, D, H, W, planes, st, guide);
  }
  size_t smem = ((size_t)cpg * (VOL_TW + UW) * gp + (size_t)Cc * (VOL_TW + UW)) * sizeof(float);
  if (smem > 220 * 1024) return DCA_ERR_UNSUPPORTED;
  const int wtiles = (W + VOL_TW - 1) / VOL_TW, dchunks = (D + VOL_DC - 1) / VOL_DC;
  dim3 grid(wtiles * dchunks, H, B);
#define DCA_VOL_LAUNCH(P, CVT)                                                                                   \
  do {                                                                                                           \
    auto kern = volume_fused_kernel<P, CVT, GT_, CPG_, GUIDED>;                                                  \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                          \
    kern<<<grid, VOL_THREADS, smem, st>>>(gwc_l, gwc_r, cat_l, cat_r, (__nv_bfloat16*)vol, B, C, G, Cc, D, H, W, Cv, \
                                          guide);                                                                \
  } while (0)
  const bool dcanet_shape = (Cv == 64 && G == 40 && cpg == 8);
#define GT_ 40
#define CPG_ 8
  if (dcanet_shape) { if (planes == 2) DCA_VOL_LAUNCH(2, 64); else DCA_VOL_LAUNCH(1, 64); }
#undef GT_
#undef CPG_
#define GT_ 0
#define CPG_ 0
  else { if (planes == 2) DCA_VOL_LAUNCH(2, 0); else DCA_VOL_LAUNCH(1, 0); }
#undef GT_
#undef CPG_
#undef DCA_VOL_LAUNCH
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
}  // namespace dca

extern "C" int dca_volume_gwc_concat(const float* gwc_l, const float* gwc_r, const float* cat_l, const float* cat_r,
                                     void* vol, int B, int C, int G, int Cc, int D, int H, int W, int Cv, int planes,
                                     void* stream) {
  return volume_gwc_concat<false>(gwc_l, gwc_r, cat_l, cat_r, vol, B, C, G, Cc, D, H, W, Cv, planes, stream,
                                  VolGuide{nullptr, 0.f, 0.f});
}

extern "C" int dca_volume_gwc_concat_guided(const float* gwc_l, const float* gwc_r, const float* cat_l,
                                            const float* cat_r, void* vol, int B, int C, int G, int Cc, int D, int H,
                                            int W, int Cv, int planes, const float* hq, float k, float s, void* stream) {
  if (!hq || !(k > 0.f) || !isfinite(k) || !(s >= 0.f) || !isfinite(s)) return DCA_ERR_ARG;
  return volume_gwc_concat<true>(gwc_l, gwc_r, cat_l, cat_r, vol, B, C, G, Cc, D, H, W, Cv, planes, stream,
                                 VolGuide{hq, k, s});
}

extern "C" int dca_build_gwc_volume_f32(const float* l, const float* r, float* vol, int B, int C, int G, int D, int H,
                                        int W, void* stream) {
  if (!l || !r || !vol || B <= 0 || C <= 0 || G <= 0 || C % G != 0 || D <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  size_t smem = (size_t)2 * (C / G) * W * sizeof(float);
  if (smem > 200 * 1024) return DCA_ERR_UNSUPPORTED;
  cudaFuncSetAttribute(gwc_volume_ncdhw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gwc_volume_ncdhw_kernel<<<dim3(H, G, B), 256, smem, (cudaStream_t)stream>>>(l, r, vol, B, C, G, D, H, W);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}

extern "C" int dca_build_concat_volume_f32(const float* l, const float* r, float* vol, int B, int C, int D, int H, int W,
                                           void* stream) {
  if (!l || !r || !vol || B <= 0 || C <= 0 || D <= 0 || H <= 0 || W <= 0) return DCA_ERR_ARG;
  size_t total = (size_t)B * 2 * C * D * H * W;
  const size_t cap = (size_t)dca_num_sms() * 16;
  int blocks = (int)((total + 255) / 256 < cap ? (total + 255) / 256 : cap);
  concat_volume_ncdhw_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(l, r, vol, B, C, D, H, W);
  DCA_RETURN_IF_LAUNCH_FAILED();
  return DCA_OK;
}
