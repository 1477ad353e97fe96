/* dca_b200.h -- C ABI of the B200 (sm_100a) DCANet cost-volume hot path.
 *
 * Drop-in boundary for everything between the 1/4-resolution feature maps and the final disparity
 * of the reference model (cocowy1/Cost-Volume-Aggregation-in-Stereo-Matching-Revisited,
 * models/gwcnet_dca_g.py:216-240).  The reference has no native code on this path (pure PyTorch
 * eager); its own precedent for this shape of boundary is models/libs/GANet/src/GANet_cuda.cpp:5-64
 * (`extern "C" int f(...)`).  Every entry point here
 *   - takes raw DEVICE pointers, sizes and a cudaStream_t (passed as void*),
 *   - never allocates, never synchronises, never throws,
 *   - returns DCA_OK (0) or a negative error code.
 * The caller (Python via ctypes, see INTEGRATION.md) owns all buffers.
 *
 * "cost planes" = channels-last 16-bit tensor [planes][B][D][H][W][C]; plane 0 = h16(x),
 * plane 1 = h16(x - plane0) (only when planes == 2, the parity precision mode); h16 = IEEE fp16 unless the library
 * was built with -DDCA_F16_PLANES=0 (bf16), see dca_plane_format().
 */
#ifndef DCA_B200_H
#define DCA_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DCA_OK 0
#define DCA_ERR_ARG (-1)         /* bad pointer / shape */
#define DCA_ERR_LAUNCH (-2)      /* CUDA launch failed */
#define DCA_ERR_UNSUPPORTED (-3) /* shape outside what the kernels were built for */

#define DCA_ACT_NONE 0
#define DCA_ACT_RELU 1
#define DCA_ACT_LEAKY 2 /* LeakyReLU(0.1) */

#define DCA_CONV_K3S1 0  /* Conv3d k3 s1 p1          (submodule.py:121-124) */
#define DCA_CONV_K3S2 1  /* Conv3d k3 s2 p1          (cva.py:16)            */
#define DCA_CONV_T3S2 2  /* ConvTranspose3d k3 s2 p1 op1 (cva.py:20-22)     */
#define DCA_CONV_K1 3    /* Conv3d 1x1x1             (cva.py:24,55)         */
#define DCA_CONV_2D3 4   /* Conv2d 3x3 s1 p1, Di==1  (gwcnet_dca_g.py:112-115) */

int dca_version(void);
/* 16-bit element format of the cost planes / tensor-core operand packs of this build: 1 = IEEE fp16 (default; hi + lo
 * = 22 significand bits), 0 = bf16 (compile with -DDCA_F16_PLANES=0; 16 bits, 8 more exponent bits). */
int dca_plane_format(void);

/* (1) volume construction -------------------------------------------------------------------- */
/* Fused replacement of build_gwc_volume (submodule.py:157-167) + build_concat_volume (:134-145)
 * + torch.cat (gwcnet_dca_g.py:220).  gwc_* [B,C,H,W] fp32, cat_* [B,Cc,H,W] fp32 (NCHW, as the
 * extractor emits them); vol = cost planes [planes][B][D][H][W][Cv], channels = G groups, Cc left,
 * Cc right, zero pad up to Cv (multiple of 8, <= 64). */
int dca_volume_gwc_concat(const float* gwc_l, const float* gwc_r, const float* cat_l, const float* cat_r, void* vol,
                          int B, int C, int G, int Cc, int D, int H, int W, int Cv, int planes, void* stream);
/* Reference-API forms: fp32 NCDHW outputs [B,G,D,H,W] / [B,2C,D,H,W]. */
int dca_build_gwc_volume_f32(const float* l, const float* r, float* vol, int B, int C, int G, int D, int H, int W,
                             void* stream);
int dca_build_concat_volume_f32(const float* l, const float* r, float* vol, int B, int C, int D, int H, int W,
                                void* stream);

/* (3) convolution family ----------------------------------------------------------------------- */
/* y = act(scale * conv(x, w) + shift + res_pre) + res_post.   CUDA-core fp32 kernel, any mode.
 * w_packed fp32 [taps][Cin][CoutPad] (dca_pack_weights); scale/shift [CoutPad] or NULL;
 * res_* cost planes shaped like y or NULL; out_kind 0 = cost planes, 1 = fp32 channels-last. */
int dca_conv3d_direct(int mode, const void* x, int planes_in, const float* w_packed, const float* scale,
                      const float* shift, const void* res_pre, const void* res_post, int planes_res, void* y,
                      int planes_out, int out_kind, int act, int B, int Cin, int Cout, int CoutPad, int Di, int Hi,
                      int Wi, int Do, int Ho, int Wo, void* stream);
/* Conv3d k3 s1 p1, Cin=32 -> 1 channel, no BN: fp32 logits [B,D,H,W] (cva.py:53, gwcnet_dca_g.py:168).
 * w_host = HOST pointer, fp32 [27][Cin]: the 864 weights travel as launch parameters (constant bank). */
int dca_conv3d_cout1(const void* x, int planes_in, const float* w_host, float* y, int B, int Cin, int D, int H, int W,
                     void* stream);
/* tcgen05/TMEM/TMA implicit-GEMM member of the family (conv_tc.cu), modes K3S1 / K3S2 / T3S2 / K1, Cin,Cout in {32,64}:
 *   y = act(scale * (conv(x, w) + trilinear_x2(up)) + shift + res_pre) + res_post
 * w_tc = bf16 operand pack from dca_pack_weights_tc; `up` (optional, Cout == 32) is a cost-plane tensor at half the
 * output resolution: the trilinear x2 + cat + 1x1x1 fuse of cva.py:64,69 folded into the epilogue.
 * `side` (optional, T3S2 only) is a cost-plane tensor [.., Do,Ho,Wo, side_c] whose 1x1x1 conv (weights = tap 27 of
 * w_tc, zero padded to Cin) joins the same GEMM: Multi_Aggregation's conv3 + redir (cva.py:20-29) in one kernel. */
int dca_conv3d_tc(int mode, const void* x, int planes_in, const void* w_tc, const float* scale, const float* shift,
                  const void* res_pre, const void* res_post, int planes_res, const void* up, int planes_up,
                  const void* side, int side_c, void* y, int planes_out, int act, int B, int Cin, int Cout, int Di,
                  int Hi, int Wi, int Do, int Ho, int Wo, void* stream);
int dca_pack_weights_tc(const float* w, int transposed, int Co, int Ci, int taps, void* out, int planes, void* stream);
long long dca_pack_weights_tc_bytes(int Co, int Ci, int taps, int planes);
/* Outputs at twice the input resolution, 8 output parity classes per low-res tile fed from shared halo slabs:
 *   kind 0: y = act(scale * (ConvTranspose3d_k3s2p1op1(x) + side 1x1x1) + shift) + res_post     (cva.py:20-29)
 *           x [planes][B][Dl][Hl][Wl][Cin]; w_tc = 27 taps (+ tap 27: side weights zero-padded to Cin)
 *   kind 1: y = act(scale * (trilinear_x2(x) + side 1x1x1) + shift) + res_post                  (cva.py:64,55,69)
 *           x = border-replicated [planes][B][Dl+2][Hl+2][Wl+2][32]; w_tc = 5 taps: {27,9,3,1}/64*I, side weights
 *   kind 2: like kind 1 but x = [planes][B][Dl][Hl+2][Wl+2][32] is already at the output depth Dl (depth axis
 *           interpolated by the producer): bilinear x2 in (h, w) only; w_tc = 4 taps {9,3,1}/16*I, side weights;
 *           side / y are [planes][B][Dl][2Hl][2Wl][..]
 * side [planes][B][2Dl][2Hl][2Wl][side_c]; Cout = 32. */
int dca_up2_tc(int kind, const void* x, int planes, const void* side, int side_c, const void* w_tc, const float* scale,
               const float* shift, const void* res_post, int planes_res, void* y, int act, int B, int Cin, int Dl,
               int Hl, int Wl, void* stream);
/* Conv3d k3 s1 p1, 32 -> 1 channel on the tensor cores: per-tap products P[tap][v] = <x[v,:], w[tap,:]> as a 1x1x1
 * GEMM (fp32, tap-major [ntap][B*D*H*W]) followed by the 27-tap shifted sum (cva.py:53, gwcnet_dca_g.py:168). */
int dca_conv1_taps_tc(const void* x, int planes, const void* w_tc, float* P, int ntap, int B, int D, int H, int W,
                      void* stream);
int dca_tap_gather3d(const float* P, float* out, int B, int D, int H, int W, void* stream);
/* Fused tail, first half: Conv3d k3 s1 p1 (Cin in {32,64} -> 32) + BN + activation whose epilogue immediately applies
 * the Conv3d(32 -> 1, k3) that follows it in classif3 (gwcnet_dca_g.py:166-168) / cva.classify (cva.py:51-53) tap by tap:
 *   P[tap][v] = sum_c w27[tap][c] * act(scale * conv(x, w)[v][c] + shift)   (fp32, tap-major [27][B*D*H*W]).
 * The 32-channel intermediate never reaches HBM.  use_march = 1: depth-marching kernel, w = dca_pack_weights_tc_march
 * pack; 0: halo-slab kernel, w = dca_pack_weights_tc pack.  w27_host is a HOST pointer ([27][32] fp32, launch params). */
int dca_conv3d_tc_taps27(const void* x, int planes, const void* w, int use_march, const float* scale, const float* shift,
                         const float* w27_host, float* P, int act, int B, int Cin, int D, int H, int W, void* stream);
/* Fused tail, second half: logits = 27-tap shifted sum of P, softmax over D, disparity regression
 * (gwcnet_dca_g.py:235-239, submodule.py:127-131): pred [B,H,W]; logits_out optional [B,D,H,W].  Neither the logits nor
 * the probability volume are materialised. */
int dca_tap_gather_softmax_regress(const float* P, float* pred, float* logits_out, int B, int D, int H, int W,
                                   void* stream);
/* Depth-marching member of the family: Conv3d k3 s1 p1, Cout = 32, Cin in {32,64}.  A CTA walks the input planes of a
 * chunk of <= 16 output planes; each halo slab is read once per (kh,kw) for all three kd (N = 96).  Same epilogue
 * contract as dca_conv3d_tc.  w_march from dca_pack_weights_tc_march ([kh*3+kw][plane][kd][32][Cin] bf16). */
int dca_conv3d_tc_march(const void* x, int planes, const void* w_march, const float* scale, const float* shift,
                        const void* res_pre, const void* res_post, int planes_res, void* y, int act, int B, int Cin,
                        int D, int H, int W, void* stream);
int dca_pack_weights_tc_march(const float* w, int Ci, void* out, int planes, void* stream);
long long dca_pack_weights_tc_march_bytes(int Ci, int planes);
/* 2-D 3x3 s1 p1 convs of the propagation net (gwcnet_dca_g.py:112-115) on the halo-slab tcgen05 kernel.
 * x [planes][B][1][H][W][Cin] (Cin 64/128); y cost planes (Cout % 64 == 0) or fp32 channels-last [B][H][W][Cout]. */
int dca_conv2d_tc(const void* x, int planes, const void* w_tc2d, const float* scale, const float* shift, void* y,
                  int out_f32, int act, int B, int Cin, int Cout, int H, int W, void* stream);
int dca_pack_weights_tc2d(const float* w, int Co, int Ci, void* out, int planes, void* stream);
long long dca_pack_weights_tc2d_bytes(int Co, int Ci, int planes);
/* The 2-D family member behind the 1/4-resolution part of the front end (SURVEY 8f-2): feature_extraction.layer2[1:],
 * layer3, layer4 (dilation 2) and lastconv (gwcnet_dca_g.py:22-29, BasicBlock submodule.py:251-273), Guidance.layer2[1],
 * conv_g0 and guidance (submodule.py:395-460, ResidualBlock :305-347).
 *   y = act_post(act(scale * conv2d_3x3(x, dilation dil) + shift) + res)
 * Cin a multiple of 64 up to 320 (64-channel slabs), dil in {1, 2} (2: H and W even; four parity sub-images through
 * strided tensor maps), res = optional cost planes shaped like y.  1x1 convs are passed as 3x3 weights whose only
 * non-zero tap is the centre. */
int dca_conv2d_tc_ex(const void* x, int planes, const void* w_tc2d, const float* scale, const float* shift,
                     const void* res, int act_post, void* y, int out_f32, int act, int B, int Cin, int Cout, int H, int W,
                     int dil, void* stream);
/* The two 3-channel stems of the front end: Conv2d(3 -> 32, K x K, stride 2, pad K/2) (+ bias) + BN + act, K in {3, 7}
 * (feature_extraction.firstconv[0] gwcnet_dca_g.py:19; Guidance.conv_start submodule.py:413-414).  x fp32 NCHW [B,3,H,W],
 * w fp32 [32][3][K][K] (torch layout), scale/shift = folded BN (+ bias); y cost planes [planes][B][1][Ho][Wo][32]. */
int dca_conv2d_stem(const float* x, const float* w, const float* scale, const float* shift, void* y, int planes, int act,
                    int B, int H, int W, int K, void* stream);
/* The same conv over the channel concatenation cat(x0, x1, x2) (each a multiple of 64 channels, <= 320 in total; unused
 * sources NULL) without materialising it: feature_extraction.lastconv on cat(l2, l3, l4) (gwcnet_dca_g.py:60-65). */
int dca_conv2d_tc_cat(const void* x0, int C0, const void* x1, int C1, const void* x2, int C2, int planes,
                      const void* w_tc2d, const float* scale, const float* shift, void* y, int out_f32, int act, int B,
                      int Cout, int H, int W, void* stream);
/* disparity groups per block of dca_tap_gather_softmax_regress (16 / 8 / 6 (default) / 4; timing experiments). */
int dca_tap_gather_set_groups(int n);
/* planes per work item of the depth-marching kernel: 0 (default) = chosen per shape (halo overhead vs fill of the last
 * wave), n > 0 = forced (timing experiments). */
int dca_tc_set_march_n(int n);
/* k3 s1 main loop selector: 1 = halo'd slab reuse (default), 0 = one TMA box per tap. */
int dca_tc_set_halo(int on);
/* bit 0 (default 1): volumes with C = 320, Cc = 12, G in {8, 20, 40} and W % 8 == 0 use the TMA-staged group-pair kernel
   (DCANet's shape is G = 40); 0: the generic kernel everywhere (A/B timing and tests).  Bits 1-2: timing probes. */
int dca_volume_set_v2(int on);
/* dca_disp_attention at D/8 == 24: 1 (default) two warps per pixel + mma.sync attention core, 2 two warps + fp32 FMA
 * core, 0 one warp per pixel (A/B timing). */
int dca_attention_set_team(int on);
/* timing probes of the tcgen05 kernels: (flags >> 4) & 1 skips the epilogue math + stores, & 2 the MMAs of the halo
 * and up2 kernels; `reserved` must be 1. */
int dca_tc_set_tuning(int reserved, int flags);
/* The tensor core truncates its fp32 accumulator toward zero at every MMA (measured: a systematic -1.56e-8 relative per
 * accumulation step).  The tcgen05 conv epilogues multiply the main accumulator block by 1 + kappa * steps; this sets
 * kappa (default 1.56e-8f, 0 = off). */
int dca_tc_set_trunc_comp(float kappa);
/* Programmatic dependent launch: 1 (default) = every kernel of the forward is launched with
 * cudaLaunchAttributeProgrammaticStreamSerialization and waits (griddepcontrol.wait) after its prologue, so prologues
 * and launch latency overlap the previous kernel's tail; 0 = plain stream order.  Same results. */
int dca_set_pdl(int on);
int dca_pdl_enabled(void);
/* dca_up2_tc kind 0 with Cin = 64 and a side input: 1 (default) = two depth-adjacent tiles per weight fetch
 * (conv_tc_deconv_pair_kernel), 0 = one tile per fetch (conv_tc_up2_kernel); same results. */
int dca_tc_set_deconv_pair(int on);
/* dca_up2_tc kind 2: depth of the side-box ring, 2 (default) or 4 (timing experiments; measured: no difference). */
int dca_tc_set_up2_side_slots(int n);

/* (2) DCA module ------------------------------------------------------------------------------- */
/* AvgPool3d(3, 2, 1) (cva.py:39).  C == 32: TMA-staged depth-marching kernel (each input plane read once); other C, or
 * after dca_pool_set_march(0): the thread-per-output kernel dca_avgpool3d_simple.  Same results (sum order differs). */
int dca_avgpool3d(const void* x, void* y, int planes, int B, int C, int Di, int Hi, int Wi, void* stream);
int dca_avgpool3d_simple(const void* x, void* y, int planes, int B, int C, int Di, int Hi, int Wi, void* stream);
int dca_pool_set_march(int on);
/* logits fp32 [B,D,H,W] -> class map int32 [B,H,W], e = exp(P[k_p]) [B,H,W], S [B,D].  S is summed in 64-bit fixed
 * point (order-independent: two runs are bit-identical); scratch = (B*D + 1) x 8 bytes, 8-byte aligned, zeroed here. */
int dca_class_stats(const float* logits, int* cls, float* e, float* S, void* scratch, int B, int D, int H, int W,
                    void* stream);
/* weights: 7 x [32][32] transposed (q0,q1,k0,k1,v,o,Wa) then 6 x (scale[32],shift[32]). */
/* pad = 1: y is [planes][B][D+2][H+2][W+2][C] with a replicated 1-voxel border (input of dca_up2_tc kind 1).
 * pad = 2: y is [planes][B][2D][H+2][W+2][C]: already interpolated x2 along depth (align_corners=False), h/w borders
 *          replicated (input of dca_up2_tc kind 2). */
int dca_disp_attention(const void* x, const int* cls, const float* e, const float* S, const float* weights,
                       int has_wa, void* y, int pad, int planes, int B, int C, int D, int H, int W, void* stream);
/* SelfAttentionBlock.forward(query_feats, key_feats) (models/augment/SelfAttention_bn.py:62-98), the generic two-input
 * form: query, key, y = cost planes [planes][B][D][H][W][32]; weights as above (the 7th matrix is not used). */
int dca_self_attention(const void* query, const void* key, const float* weights, void* y, int planes, int B, int C,
                       int D, int H, int W, void* stream);
/* y = scale * (trilinear_x2(t) + WcT^T cost) + shift ; t at (Dl,Hl,Wl), cost / y at twice that. */
int dca_upsample_fuse(const void* t, const void* cost, const float* WcT, const float* scale, const float* shift,
                      void* y, int planes, int B, int C, int Dl, int Hl, int Wl, void* stream);

/* (4) regression + convex upsampling ------------------------------------------------------------ */
int dca_softmax_regress(const float* logits, float* pred, int B, int D, int H, int W, void* stream);
/* disparity_regression on its own (models/submodule.py:127-131): pred[b,h,w] = sum_d d * x[b,d,h,w], x not renormalised. */
int dca_regress_f32(const float* x, float* pred, int B, int D, int H, int W, void* stream);
int dca_convex_upsample(const float* mask, const float* disp, float* out, int B, int H, int W, void* stream);
/* Per-pixel confidence of the disparity, from the classif head's logits l[d] [B,D,H,W] (D = D4 = maxdisp / 4) at 1/4 res.
 * With p = softmax_d(l) and mu = sum_d d p(d) (= pred_quarter):
 *   peak_q = max_d p(d)                          in [1/D, 1]
 *   std_q  = sqrt(sum_d p(d) (d - mu)^2)         in 1/4-res disparity units; computed in centred form (max, then sum
 *                                                and mean, then the centred second moment: three passes over the logits),
 *                                                never as E[d^2] - mu^2, which in fp32 at D = 48 loses ~0.05 px on confident
 *                                                pixels
 * At full resolution both maps are convex-upsampled with the 9-neighbour softmax weights of `mask` (the prop net's fp32
 * channels-last [B,H,W,144], as dca_convex_upsample) and the same zero padding outside the image as pred4:
 *   peak = up(peak_q) in [0, 1],  std = up(4 std_q) in full-res px.
 * The upsampled std is a convex combination of the neighbouring stds, not the std of the mixture of their distributions.
 * The zero padding lowers the confidence along the image border (peak toward 0, std toward 0), exactly where pred4 is
 * pulled toward 0 by the same padding.
 * A CTA owns a 32 x 8 tile of 1/4-res pixels and recomputes the statistics of its 1-pixel ring (as
 * dca_softmax_regress_upsample).  peak_q / std_q [B,H,W] are optional (NULL = not written); peak / std [B,1,4H,4W]. */
int dca_softmax_confidence_upsample(const float* logits, const float* mask, float* peak_q, float* std_q, float* peak,
                                    float* std, int B, int D, int H, int W, void* stream);

/* (5) H-sharded single-pair mode: halo rows over NVLink peer memory ------------------------------ */
/* Replaces, for BASELINE configs[4] (one pair row-sharded over the GPUs of a box, SURVEY section 8e), the exchange a
 * multi-GPU port of the reference would do with NCCL send/recv after every 3x3x3 layer.  `t` is viewed as
 * [outer][rows][inner_bytes]; the rank owns rows [h, rows-h) and only the `live` <= h halo rows next to them are ever read.
 * dca_halo_push stores the owned rows [h,h+live) / [rows-h-live,rows-h) into the upper / lower neighbour's staging slot (peer-mapped addresses, 0 = no neighbour) and bumps the neighbour's
 * 64-bit arrival counter by dca_halo_push_ctas(); dca_halo_wait_unpack spins (bounded: dca_halo_set_timeout_ms, default 10 s, then *err = 1) until the
 * own counters reach `target` and copies the staged rows into the halo rows [h-live,h) / [rows-h,rows-h+live).  Needs 16-byte aligned rows
 * (DCA_ERR_UNSUPPORTED otherwise: use the NCCL transport for that tensor). */
int dca_halo_push_ctas(void);
int dca_halo_set_timeout_ms(int ms);
int dca_halo_push(const void* t, long long outer, long long rows, long long inner_bytes, int h, int live, void* peer_up_stage,
                  void* peer_down_stage, void* peer_up_flag, void* peer_down_flag, void* stream);
int dca_halo_wait_unpack(void* t, long long outer, long long rows, long long inner_bytes, int h, int live,
                         const void* stage_top,
                         const void* stage_bottom, const void* flag_top, const void* flag_bottom,
                         unsigned long long target, void* err, void* stream);

/* the two calls above as ONE launch (same arguments and semantics): what hshard.PeerHalo issues per exchange */
int dca_halo_exchange(void* t, long long outer, long long rows, long long inner_bytes, int h, int live,
                      void* peer_up_stage, void* peer_down_stage, void* peer_up_flag, void* peer_down_flag,
                      const void* stage_top, const void* stage_bottom, const void* flag_top, const void* flag_bottom,
                      unsigned long long target, void* err, void* stream);

/* (6) compositions under the family names of SURVEY.md section 8(b) -------------------------------- */
/* dca_conv3d_igemm: the implicit-GEMM family (convbn_3d / Conv3d s2 / ConvTranspose3d / 1x1x1, submodule.py:121-124,
 * cva.py:16-24): same contract as dca_conv3d_tc. */
int dca_conv3d_igemm(int mode, const void* x, int planes_in, const void* w_tc, const float* scale, const float* shift,
                     const void* res_pre, const void* res_post, int planes_res, const void* up, int planes_up,
                     const void* side, int side_c, void* y, int planes_out, int act, int B, int Cin, int Cout, int Di,
                     int Hi, int Wi, int Do, int Ho, int Wo, void* stream);
/* dca_pool_conv: cva.downsample (cva.py:39-41) = dca_avgpool3d into the caller's `pooled` scratch, then the 3x3x3 conv +
 * folded BN + act on it; y and pooled are [planes][B][(Di+1)/2][(Hi+1)/2][(Wi+1)/2][C]. */
int dca_pool_conv(const void* x, void* pooled, const void* w_tc, const float* scale, const float* shift, void* y,
                  int planes, int act, int B, int C, int Di, int Hi, int Wi, void* stream);
/* dca_softmax_regress_upsample: gwcnet_dca_g.py:238-239 + :117-124 in ONE kernel: softmax over D + disparity regression
 * of a 32 x 8 pixel tile and its 1-pixel ring into shared memory, convex 4x upsampling from there.  pred_q [B,1,H,W] =
 * the 1/4-res disparity, out [B,1,4H,4W].  Bit-identical to dca_softmax_regress + dca_convex_upsample. */
int dca_softmax_regress_upsample(const float* logits, const float* mask, float* pred_q, float* out, int B, int D, int H,
                                 int W, void* stream);

/* F.adaptive_avg_pool3d(x[:, :, h0:, :], (Do, Ho, Wo)) of an fp32 [B][D][H][W] tensor: the `vis_tsne1` head of the
 * plain-GwcNet baseline (models/gwcnet.py:186-190). */
int dca_adaptive_avgpool3d_rows(const float* x, float* y, int B, int D, int H, int W, int h0, int Do, int Ho, int Wo,
                                void* stream);

/* (7) accuracy against ground-truth disparity: the evaluation loop of main_dca.py `mytest` (:143-232) ------------------ */
/* Both kernels ADD into caller-zeroed 64-bit counters (integer sums: bit-reproducible in any launch order), never
 * allocate or synchronise, and may be captured in a CUDA graph.  A GT pixel g is valid when
 *   isfinite(g) && g > 0 && (max_valid <= 0 || g < max_valid)
 * (the SceneFlow mask (gt > 0) & (gt < maxdisp) of the GwcNet / PSMNet test loops; KITTI's 0 and Middlebury's inf are
 * invalid).  All arithmetic is IEEE fp32 without fast math. */
#define DCA_METRIC_VALID 0         /* valid GT pixels */
#define DCA_METRIC_SUM_ABS 1       /* sum over valid pixels with a finite prediction of E = |pred - gt|, in units of 2^-20 px:
                                      min(E, 2^20) * 2^20 rounded to nearest-even.  Each pixel adds <= 2^40, so a row is exact
                                      (no overflow) while the valid pixels added into it number at most 2^23. */
#define DCA_METRIC_GT1 2           /* valid pixels with E > 1 */
#define DCA_METRIC_GT2 3           /* valid pixels with E > 2 */
#define DCA_METRIC_GT3 4           /* valid pixels with E > 3 */
#define DCA_METRIC_D1 5            /* valid pixels with E > 3 && E / |gt| > 0.05f (GwcNet D1_metric, division form) */
#define DCA_METRIC_PRED_NONFINITE 6 /* valid pixels whose prediction is NaN or inf: counted in GT1..D1, not in SUM_ABS */
#define DCA_METRIC_COUNT 7
/* pred, gt fp32 [B,H,W] in the same pixel frame (pred4 [B,1,H,W] is the same memory); rows [B][DCA_METRIC_COUNT]:
 * rows[b][m] += counter m of image b.  B <= 65535. */
int dca_disparity_metrics(const float* pred, const float* gt, unsigned long long* rows, int B, int H, int W,
                          float max_valid, void* stream);
/* Confusion matrix of the DCA disparity classes (main_dca.py:66-120, 209-232): logits fp32 [B,D8,H8,W8] (prob_volume2),
 * gt fp32 [B,8*H8,8*W8] in the same frame; conf [D8][D8] += pixel count, row = GT class, column = predicted class.
 * Predicted class = first argmax of the fp32 softmax, exactly as dca_class_stats.  GT class of 1/8-res pixel (i, j):
 * g = gt[8i, 8j] (F.interpolate(gt, scale_factor=1/8, mode='nearest')), valid as above, class
 * min(floorf(g * 0.125f + 0.5f), D8 - 1) = the nearest 1/8-res disparity plane (plane k is centred on 8k px).  This GT
 * rule is this library's definition: the reference's own rule is not pinned by any fixture.  D8 <= 64. */
int dca_class_confusion(const float* logits, const float* gt, unsigned long long* conf, int B, int D8, int H8, int W8,
                        float max_valid, void* stream);
/* Sparsification tables of a confidence map: pred, gt, peak fp32 [B,H,W] in the same pixel frame (peak = the full-res
 * confidence of dca_softmax_confidence_upsample).  Over exactly the pixels that enter DCA_METRIC_SUM_ABS (valid GT, finite
 * prediction), with F = the per-pixel fixed-point |E| of SUM_ABS:
 *   conf_hist [DCA_CONF_BINS][2] += (1, F) at bin min(floorf(peak * 256), 255); a NaN, inf or negative peak -> bin 0
 *   err_hist  [DCA_ERR_BINS][2]  += (1, F) at bin min(F >> 15, 2048): 1/32 px bins over [0, 64), the last one E >= 64
 * Sums over either table equal SUM_ABS / (VALID - PRED_NONFINITE) of dca_disparity_metrics on the same inputs.  Integer
 * sums, exact while they stay below 2^64 (E < 512 px: 2^35 pixels). */
#define DCA_CONF_BINS 256
#define DCA_ERR_BINS (2048 + 1)
int dca_confidence_histograms(const float* pred, const float* gt, const float* peak, unsigned long long* conf_hist,
                              unsigned long long* err_hist, int B, int H, int W, float max_valid, void* stream);
/* Depth errors of the Eigen et al. protocol (monodepth, pseudo-LiDAR) for a batch that shares one calibration,
 * fB = focal_baseline (fx B, metres x px) and doffs (px), all in IEEE fp32:
 *   pixels   valid GT as above, with Zg = fB / (gt + doffs) and min_depth <= Zg <= max_depth
 *   Zp       fB / (pred + doffs), or max_depth when pred + doffs is not finite or <= 0; then clamped into
 *            [min_depth, max_depth]
 * rows [B][DCA_DEPTH_COUNT] += the counters of image b.  The four sums are fixed point like DCA_METRIC_SUM_ABS: each
 * per-pixel term t is added as min(t, 2^20) * 2^20 rounded to nearest-even (unit 2^-20 of the term's unit), so a pixel
 * adds <= 2^40 and a row is exact while it holds at most 2^23 valid pixels.  DCA_ERR_ARG for NULL pointers, B, H, W <= 0,
 * B > 65535, a NaN max_valid, fB <= 0 or not finite, a non-finite doffs, min_depth <= 0 and max_depth not finite or
 * < min_depth; DCA_ERR_UNSUPPORTED for H W > 2^31 - 257. */
#define DCA_DEPTH_VALID 0      /* pixels scored */
#define DCA_DEPTH_ABS_REL 1    /* sum |Zp - Zg| / Zg                   (unit 2^-20) */
#define DCA_DEPTH_SQ_REL 2     /* sum (Zp - Zg)^2 / Zg                 (unit 2^-20 m) */
#define DCA_DEPTH_SQ 3         /* sum (Zp - Zg)^2                      (unit 2^-20 m^2) */
#define DCA_DEPTH_LOG_SQ 4     /* sum (ln Zp - ln Zg)^2 (logf)         (unit 2^-20) */
#define DCA_DEPTH_A1 5         /* pixels with max(Zp / Zg, Zg / Zp) < 1.25 */
#define DCA_DEPTH_A2 6         /* ... < 1.25^2 */
#define DCA_DEPTH_A3 7         /* ... < 1.25^3 */
#define DCA_DEPTH_COUNT 8
int dca_depth_metrics(const float* pred, const float* gt, unsigned long long* rows, int B, int H, int W,
                      float max_valid, float focal_baseline, float doffs, float min_depth, float max_depth,
                      void* stream);

/* (8) left-right consistency check and background fill ------------------------------------------------------------- */
/* Right view.  DCANet is not mirror-symmetric (the guidance comes from the left image, the volume is built with the left
 * image as reference), so the right view's disparity comes from the mirror trick: with flip = mirror of the W axis,
 *   D_R = flip(net(flip(R), flip(L)))
 * (the swapped, mirrored pair is again a left-referenced problem with positive disparities).
 * Check of left pixel (y, x) with d = D_L(y, x), all in fp32 with explicit rounding (no contraction):
 *   xr = x - d
 *   not 0 <= xr <= W-1 (a non-finite d included)                                     -> DCA_LR_OUT_OF_VIEW
 *   x0 = floor(xr), a = xr - x0;  v = D_R[x0] if x0 == W-1, else D_R[x0] + a * (D_R[x0+1] - D_R[x0])
 *   |d - v| <= tau                                                                   -> DCA_LR_CONSISTENT
 *   else v - d > tau (the right view sees a nearer surface there)                    -> DCA_LR_OCCLUDED
 *   else (a non-finite v included)                                                   -> DCA_LR_MISMATCH
 * Background fill, one row at a time: a consistent pixel keeps D_L; any other pixel takes min(D_L[l], D_L[r]) with l / r
 * the nearest consistent pixels to its left / right on the same row, the one that exists when only one does, and D_L
 * when the row has no consistent pixel.  This is the background fill of occlusion handling; mismatches are filled the
 * same way on purpose, to keep the rule simple.
 * disp_left, disp_right fp32 [B,H,W] (pred4 [B,1,H,W] is the same memory); right_mirrored != 0 reads disp_right in the
 * layout of the mirrored forward (disp_right[b, y, W-1-x] = D_R(y, x)), so no flipped copy is needed.  Outputs [B,H,W]:
 * label uint8 (DCA_LR_*), filled fp32, and disp_right_out (NULL = not written) the un-mirrored D_R.  One CTA per
 * (image, row) stages a row in shared memory, 9 bytes per pixel: W <= DCA_LR_MAX_W keeps that under the 48 KB a CTA gets
 * without an opt-in (DCA_ERR_UNSUPPORTED above).  DCA_ERR_ARG for NULL required pointers, B, H, W <= 0, B > 65535, and a
 * tau that is NaN or negative. */
#define DCA_LR_CONSISTENT 0
#define DCA_LR_OCCLUDED 1
#define DCA_LR_MISMATCH 2
#define DCA_LR_OUT_OF_VIEW 3
#define DCA_LR_MAX_W 4096
int dca_lr_consistency(const float* disp_left, const float* disp_right, int right_mirrored, unsigned char* label,
                       float* filled, float* disp_right_out, int B, int H, int W, float tau, void* stream);

/* (9) metric depth and 3-D points: reprojection of a disparity window ------------------------------------------------ */
/* Pixel (y, x) of an H x W window, with d = disp, all in fp32 with explicit rounding (no contraction), each matrix row
 * applied as ((m0 a + m1 b) + m2 c) + m3:
 *   u = x + u0, v = y + v0 (exact)
 *   (X', Y', Z', W') = Q (u, v, d, 1),  X = X' / W', Y = Y' / W', Z = Z' / W'   (OpenCV's reprojectImageTo3D convention;
 *                                       for a rectified pair Q = [[1,0,0,-cx],[0,fx/fy,0,-cy fx/fy],[0,0,0,fx],
 *                                       [0,0,1/B,doffs/B]] gives Z = fx B / (d + doffs))
 * The pixel is KEPT iff d is finite, W' > 0, min_depth <= Z <= max_depth, (peak == NULL or peak >= min_peak) and
 * (label == NULL or label == DCA_LR_CONSISTENT).  A kept pixel appends P = T (X, Y, Z, 1) ((X, Y, Z) when T is NULL) to
 * xyz[b], its window index y W + x to index[b], and sets depth[b, y, x] = Z (camera-frame Z, before T); any other pixel
 * sets depth[b, y, x] = 0 (KITTI's "no depth") and appends nothing.  Points are in row-major pixel order whatever the
 * scheduling; count[b] = the number kept, rows of xyz[b] / index[b] past it are not written.
 * disp, peak (fp32, optional) and label (uint8 DCA_LR_*, optional) share one layout: element (b, y, x) at
 * b pitch_img + y pitch_row + x, so a cropped view of pred4 needs no copy.  Q_host [4][4] and T_host [3][4] (or NULL) are
 * HOST pointers, row-major, that travel as launch parameters.  Outputs: depth fp32 [B,H,W] (NULL = not written),
 * xyz fp32 [B][H W][3], index int32 [B][H W], count int64 [B]; workspace int32 [B][ceil(H W / DCA_REPROJECT_TILE)]
 * holds the per-tile counts between the two launches (count, then an ordered scatter; no CTA waits on another).
 * DCA_ERR_ARG for NULL required pointers, B, H, W <= 0, B > 65535, H W >= 2^31, pitch_row < W, pitch_img < H pitch_row,
 * a NaN min_peak / min_depth / max_depth and min_depth > max_depth. */
#define DCA_REPROJECT_TILE 1024
int dca_reproject(const float* disp, const float* peak, const unsigned char* label, long long pitch_row,
                  long long pitch_img, int B, int H, int W, int u0, int v0, const float* Q_host, const float* T_host,
                  float min_peak, float min_depth, float max_depth, float* depth, float* xyz, int* index,
                  long long* count, int* workspace, void* stream);

/* (10) rectification of raw stereo pairs and the standardised network input -------------------------------------- */
/* dca_rectify.  maps fp32 [2][H][W][2] (view 0 = left, 1 = right): the source coordinate (sx, sy) of rectified pixel
 * (y, x), pixel centres at integer coordinates (OpenCV's initUndistortRectifyMap convention, built once on the host).
 * Per rectified pixel, view and channel c = 0..2, all in fp32 with explicit rounding (no contraction):
 *   x0 = floorf(sx), ax = sx - x0, y0 = floorf(sy), ay = sy - y0
 *   p00, p01, p10, p11 = the source bytes at (x0, y0), (x0+1, y0), (x0, y0+1), (x0+1, y0+1); a tap outside the source
 *                        image is 0 (OpenCV's BORDER_CONSTANT, value 0); a non-finite sx or sy gives v = 0
 *   v = (1-ay) ((1-ax) p00 + ax p01) + ay ((1-ax) p10 + ax p11), evaluated as written: each product rounded, then each
 *       sum, (1-a) rounded first
 *   q = clamp(rint(v), 0, 255)   (round half to even: __float2int_rn)
 * Rounding to uint8 is deliberate: the result is what rectifying to a PNG and loading it gives, and the moments below are
 * exact integers.  It is NOT bit-compatible with cv2.remap, which quantises the map to 1/32 px.
 * Sources: left / right uint8 [B][Hs][Ws][channels], channels 3 (RGB) or 4 (RGBA, channel 3 unused); byte (b, y, x, c) at
 * b pitch_img + y pitch_row + x channels + c, so a strided view or a pinned slot needs no copy.  Outputs: rgb uint8
 * [B][2][H][W][3] (HWC, view 0 = left), and moments uint64 [B][2][3][2] += (sum q, sum q^2) of each image and channel;
 * the caller zeroes moments.  Each CTA adds its 32-bit sums with one integer atomic per counter, so the totals are
 * exact and deterministic.  One CTA per DCA_RECTIFY_TILE rectified pixels of one image.
 *
 * dca_standardise_frame.  Per image and channel, with N = H W, S = sum q, SS = sum q^2 from moments:
 *   mean = S / N                                   fp64, correctly rounded (numpy's mean of the uint8 channel)
 *   var  = fp64(N SS - S^2) / (fp64(N) fp64(N))    the numerator exact in 128-bit integers, then correctly rounded to
 *                                                  fp64; the denominator one fp64 product; one fp64 division
 *   std  = sqrt(var)                               fp64, correctly rounded
 *   out  = fp32((q - mean) / std)                  fp64 subtraction and division, one rounding to fp32 (a constant
 *                                                  channel gives NaN, as kitti_io.load_pair does)
 * Framing: outputs left / right fp32 [B][3][Hn][Wn] (two tensors, NCHW); frame pixel (yn, xn) with
 * dst_y0 <= yn < dst_y0 + win_h and xn < win_w takes rectified pixel (yn - dst_y0 + src_y0, xn), every other frame pixel
 * is 0.  kitti_io.fit_to_crop of a smaller image is (Hn, Wn) = (crop_h, crop_w), dst_y0 = crop_h - H, src_y0 = 0,
 * window H x W; of a larger one dst_y0 = 0, src_y0 = int((H - crop_h) / 2), window crop_h x crop_w; pad_to_multiple(16)
 * is Hn, Wn = H, W rounded up to 16, dst_y0 = Hn - H, src_y0 = 0, window H x W.
 *
 * Both: DCA_ERR_ARG for NULL pointers, sizes <= 0, B > 65535, channels other than 3 or 4, pitch_row < Ws channels,
 * pitch_img < Hs pitch_row, and a copy window outside the frame or the rectified image; DCA_ERR_UNSUPPORTED for
 * H W, Hs Ws or Hn Wn >= 2^31 and Hs or Ws > 2^24. */
#define DCA_RECTIFY_TILE 1024
int dca_rectify(const unsigned char* left, const unsigned char* right, int channels, long long pitch_row,
                long long pitch_img, int B, int Hs, int Ws, const float* maps, int H, int W, unsigned char* rgb,
                unsigned long long* moments, void* stream);
int dca_standardise_frame(const unsigned char* rgb, const unsigned long long* moments, int B, int H, int W, float* left,
                          float* right, int Hn, int Wn, int dst_y0, int src_y0, int win_h, int win_w, void* stream);

/* (11) edge-aware refinement: confidence-weighted fast global smoother guided by the left image ------------------- */
/* The fast global smoother of Min et al. (IEEE TIP 2014), the solver inside OpenCV's ximgproc DisparityWLSFilter.  The
 * result is NOT bit-compatible with OpenCV's implementation (different weights, schedule rounding and solve order).
 * Pixel p = (b, y, x) of an H x W window, all in fp32 with explicit rounding (no contraction); (+) (-) (x) (/) are the
 * correctly rounded fp32 operations:
 *   c = clamp(peak, 0, 1), 0 for a NaN peak, 1 without peak;  c = 0 where label != DCA_LR_CONSISTENT (with label) and
 *       where d = disp is not finite
 *   U = c (x) d where c > 0, else 0 (a non-finite d never enters);  V = c
 *   w(p, q) = lut[sum over the channels 0..2 of (g_p - g_q)^2] for horizontal and vertical neighbours p, q (the sum is an
 *       exact integer <= 3 255^2); lut[k] = fp32(exp(-sqrt(k) / sigma)) built in float64 on the host, so no
 *       transcendental function runs on the device
 *   for t = 1..T: lambda_t = fp32(((lambda 1.5) 4^(T-t)) / (4^T - 1)) in float64 (the FGS schedule, OpenCV's
 *       lambda_attenuation = 0.25), computed by this entry point on the host; then one pass over every row (lines of
 *       n = W along x), then one pass over every column (lines of n = H along y).  A pass solves, on each line, for U and
 *       for V with the same matrix,
 *         (1 + e_{i-1} + e_i) u_i - e_{i-1} u_{i-1} - e_i u_{i+1} = f_i,   e_i = lambda_t (x) w(i, i+1),
 *         e_{-1} = e_{n-1} = 0,   b_i = (1 (+) e_{i-1}) (+) e_i
 *       partitioned as follows (K = DCA_WLS_SEGMENT).  The separators are the elements c = K-1, 2K-1, ... with
 *       c <= n-2; they split the line into S = DCA_WLS_SEGMENTS(n) segments [a, c) of 1..K elements (a = 0 or one past a
 *       separator, c = the next separator or n), with eL = e_{a-1} (0 for a = 0) and eR = e_{c-1}.
 *       THOMAS(f) of a segment, Thomas elimination in reciprocal form with e_{a-1} = eL, p = g = 0 before a, u = 0 at c:
 *         forward  i = a..c-1:  m_i = 1 (/) (b_i (-) e_{i-1} (x) p_{i-1})
 *                               p_i = e_i (x) m_i
 *                               g_i = (f_i (+) e_{i-1} (x) g_{i-1}) (x) m_i
 *         backward i = c-1..a:  u_i = g_i (+) p_i (x) u_{i+1}
 *       (1) boundary values of each segment (only when S > 1), for U and V:
 *           last element:  y_last = g_{c-1} of the forward sweep on f;  phi_last = G_{c-1} with G_a = eL (x) m_a,
 *                          G_i = (e_{i-1} (x) G_{i-1}) (x) m_i;  psi_last = eR (x) m_{c-1}
 *           first element: the reverse sweep i = c-1..a with r = h = 0 after c-1:
 *                          q_i = 1 (/) (b_i (-) e_i (x) r_{i+1}),  r_i = e_{i-1} (x) q_i,
 *                          h_i = (f_i (+) e_i (x) h_{i+1}) (x) q_i;  y_first = h_a;  phi_first = eL (x) q_a;
 *                          psi_first = Q_a with Q_{c-1} = eR (x) q_{c-1}, Q_i = (e_i (x) Q_{i+1}) (x) q_i
 *       (2) the separators x_0..x_{S-2} (x_s at c_s = (s+1) K - 1, between segments s and s+1), for U and V:
 *           lo_s = e_{c-1} (x) phi_last(s),  up_s = e_c (x) psi_first(s+1),
 *           D_s = (b_c (-) e_{c-1} (x) psi_last(s)) (-) e_c (x) phi_first(s+1),
 *           r_s = (f_c (+) e_{c-1} (x) y_last(s)) (+) e_c (x) y_first(s+1);
 *           forward s = 0..S-2 with P = G = 0 before 0:  M = 1 (/) (D_s (-) lo_s (x) P_{s-1}),  P_s = up_s (x) M,
 *           G_s = (r_s (+) lo_s (x) G_{s-1}) (x) M;  backward with x_{S-1} = 0:  x_s = G_s (+) P_s (x) x_{s+1}
 *       (3) each segment: THOMAS(f') with f' = f except f'_a = f_a (+) eL (x) x_{s-1} when a > 0, then
 *           f'_{c-1} = f'_{c-1} (+) eR (x) x_s when c < n (in that order when a = c-1)
 *       The solution (the separators' x, the segments' u) replaces f.  With S = 1 (n <= K) the pass is THOMAS(f) on
 *       the whole line.
 *   support = V after the last pass: in [0, 1] up to the rounding of the fp32 solves (the exact solve averages, so a
 *       pixel far from any confident pixel gets a small support);  refined = U (/) V where V >= min_support, else disp
 * min_support = 0 makes 0 / 0 = NaN possible where V = 0; the default of the Python wrapper is 1e-3, because where
 * every path to a confident pixel crosses strong colour edges V underflows towards the denormals and U / V loses all
 * precision (DESIGN.md, "Refinement").
 * disp, peak (fp32, optional) and label (uint8 DCA_LR_*, optional) share one layout: element (b, y, x) at
 * b pitch_img + y pitch_row + x, so a cropped view of pred4 needs no copy.  guide uint8 [B][H][W][channels], channels
 * 3 (RGB) or 4 (RGBA, channel 3 unused): byte (b, y, x, c) at b guide_pitch_img + y guide_pitch_row + x channels + c.
 * lut fp32 [DCA_WLS_LUT_SIZE] on the device.  Outputs refined, support fp32 [B,H,W] (contiguous; they hold U and V
 * between the passes).  workspace = DCA_WLS_WORKSPACE_BYTES(B, H, W) bytes: the horizontal and vertical weights and 8
 * boundary values per segment of each pass.  A pass is 3 launches (1 when its lines have no separator), so a call is
 * at most 1 + 6T; no host sync, no allocation: capturable in a CUDA graph.  DCA_ERR_ARG for NULL required pointers,
 * B, H, W <= 0, B > 65535, channels other than 3 or 4, pitch_row < W, pitch_img < H pitch_row,
 * guide_pitch_row < W channels, guide_pitch_img < H guide_pitch_row, num_iter outside 1..DCA_WLS_MAX_ITER, a lambda that
 * is NaN, infinite or negative and a NaN or negative min_support; DCA_ERR_UNSUPPORTED for H W >= 2^31 and for more
 * than 65535 segments per line (H or W > 65535 K). */
#define DCA_WLS_LUT_SIZE (3 * 255 * 255 + 1)
#define DCA_WLS_MAX_ITER 8
#define DCA_WLS_SEGMENT 64
#define DCA_WLS_SEGMENTS(n) (((n) - 1) / DCA_WLS_SEGMENT + 1)
#define DCA_WLS_WORKSPACE_BYTES(B, H, W)                                                                              \
  (4ull * (unsigned long long)(B) *                                                                                   \
   (2ull * (unsigned long long)(H) * (unsigned long long)(W) +                                                        \
    8ull * ((unsigned long long)(H) * DCA_WLS_SEGMENTS((unsigned long long)(W)) +                                     \
            (unsigned long long)(W) * DCA_WLS_SEGMENTS((unsigned long long)(H)))))
int dca_wls_filter(const float* disp, const float* peak, const unsigned char* label, long long pitch_row,
                   long long pitch_img, int B, int H, int W, const unsigned char* guide, int channels,
                   long long guide_pitch_row, long long guide_pitch_img, const float* lut, float lambda, int num_iter,
                   float min_support, float* refined, float* support, void* workspace, void* stream);

/* (12) TSDF fusion of posed depth maps and the surface of the fused volume ----------------------------------------- */
/* Curless & Levoy (SIGGRAPH 1996) in the projective form of KinectFusion (Newcombe et al., ISMAR 2011), on a dense grid.
 * All in fp32 with explicit rounding (no contraction); (+) (-) (x) (/) are the correctly rounded fp32 operations and each
 * matrix row is applied as ((m0 a (+) m1 b) (+) m2 c) (+) m3.
 * Volume: nx x ny x nz voxels; voxel (i, j, k) has linear index v = (k ny + j) nx + i (x fastest) and centre
 * p = (ox (+) vs (x) fp32(i), oy (+) vs (x) fp32(j), oz (+) vs (x) fp32(k)) in world metres.  State: planar fp32 with
 * plane stride N = nx ny nz, plane 0 = tsdf T (initialised to 1), 1 = weight W (initialised to 0), 2..4 = colour r, g, b
 * (initialised to 0; planes = 5) or no colour (planes = 2).  The caller initialises the state.
 *
 * dca_tsdf_integrate.  Only the voxels of the box i0..i0+bi-1, j0..j0+bj-1, k0..k0+bk-1 are read or written.  Per voxel,
 * the state is held in registers while the frames b = 0..B-1 are applied in order (so one call with B frames equals B
 * calls with one frame each, bit for bit); frame b is skipped at the first failing step:
 *   (Xc, Yc, Zc) = T_b p, with T_b = T_host[b] the world-to-camera 3x4 (row-major);  skip unless Zc > 0
 *   x = ((fx (x) Xc) (/) Zc) (+) cx (-) fp32(u0),  y = ((fy (x) Yc) (/) Zc) (+) cy (-) fp32(v0)
 *   xf = floorf(x (+) 0.5), yf = floorf(y (+) 0.5);  skip unless 0 <= xf < W and 0 <= yf < H (in float, so NaN skips)
 *   z = depth[b, yf, xf];  skip unless z is finite and 0 < z <= max_depth
 *   w = the observation weight: 1 without a weight map, else the map clamped to [0, 1], 0 where it holds NaN;
 *       skip unless w > 0
 *   sdf = z (-) Zc;  skip if sdf < -trunc;  f = min(1, sdf (/) trunc)
 *   Wn = W (+) w;  T = ((T (x) W) (+) (f (x) w)) (/) Wn;  with colour, for c = r, g, b with q = fp32 of the pixel's byte
 *       C = ((C (x) W) (+) (q (x) w)) (/) Wn;  then W = min(Wn, max_weight)
 * A voxel that no frame updates is left as it was.  depth (and weight, optional) fp32: element (b, y, x) at
 * b pitch_img + y pitch_row + x (window pixel (x, y) is image pixel (x + u0, y + v0), as in dca_reproject).  rgb uint8
 * [B][H][W][channels], channels 3 (RGB) or 4 (RGBA, channel 3 unused): byte (b, y, x, c) at
 * b rgb_pitch_img + y rgb_pitch_row + x channels + c; it is required with planes = 5 and must be NULL with planes = 2.
 * T_host [B][12] is a HOST pointer that travels as launch parameters.  One launch, no atomics, no host sync, no
 * allocation: capturable in a CUDA graph.
 * DCA_ERR_ARG for NULL volume / depth / T_host, planes other than 2 or 5, nx, ny, nz, H, W <= 0, B outside
 * 1..DCA_TSDF_MAX_FRAMES, pitch_row < W, pitch_img < H pitch_row, an rgb given or missing against planes, channels other
 * than 3 or 4, rgb_pitch_row < W channels, rgb_pitch_img < H rgb_pitch_row, a box that is empty or leaves the grid, NaN
 * ox / oy / oz / fx / fy / cx / cy / max_depth, voxel_size, trunc or max_weight not > 0 (max_weight = inf: no cap);
 * DCA_ERR_UNSUPPORTED for N >= 2^31, H or W >= 2^24 and |u0| or |v0| >= 2^24.
 *
 * Surface crossings.  For voxel v and axis a in (x, y, z) whose neighbour n = v + e_a lies inside the grid, there is a
 * crossing when W(v) >= min_weight, W(n) >= min_weight and (T(v) < 0) != (T(n) < 0).  Its point is p(v) with component
 * a replaced by p_a(v) (+) (t (x) vs), t = T(v) (/) (T(v) (-) T(n)).  Points are ordered by v, then by axis x, y, z.
 *   normal: g = (T(i+1) (-) T(i-1), T(j+1) (-) T(j-1), T(k+1) (-) T(k-1)) at v, each neighbour index clamped into the
 *           grid; len = __fsqrt_rn((gx (x) gx (+) gy (x) gy) (+) gz (x) gz); g (/) len, or (0, 0, 0) when len = 0.  It
 *           points from negative (behind the surface) to positive (towards the cameras).
 *   colour: per channel clamp(rint(C(v) (+) t (x) (C(n) (-) C(v))), 0, 255) (round half to even), uint8.
 * dca_tsdf_count_surface writes the crossings of each tile of DCA_TSDF_TILE voxels (in linear index order) to
 * workspace int64 [ceil(N / DCA_TSDF_TILE)], then, in one CTA, replaces them by their exclusive prefix sums (each tile's
 * first output row) and writes the total to count (int64, device).  dca_tsdf_extract_surface, on the same volume and
 * min_weight after it, recomputes the crossings of each tile and writes rows o < capacity: xyz fp32 [capacity][3],
 * normal fp32 [capacity][3] (NULL = not written), rgb uint8 [capacity][3] (NULL = not written; planes = 5 only).  count
 * keeps the true total, so a caller sees a truncated extraction.  Three launches in all, no atomics, no CTA waits on
 * another.  DCA_ERR_ARG for a NULL volume / workspace / count, planes other than 2 or 5, nx, ny, nz <= 0, a NaN
 * min_weight, NaN ox / oy / oz, voxel_size not > 0, capacity < 0, a NULL xyz with capacity > 0 and rgb with planes = 2;
 * DCA_ERR_UNSUPPORTED for N >= 2^31. */
#define DCA_TSDF_MAX_FRAMES 16
#define DCA_TSDF_TILE 1024
int dca_tsdf_integrate(float* volume, int planes, int nx, int ny, int nz, float ox, float oy, float oz,
                       float voxel_size, int i0, int j0, int k0, int bi, int bj, int bk, const float* depth,
                       const float* weight, long long pitch_row, long long pitch_img, int B, int H, int W,
                       const unsigned char* rgb, int channels, long long rgb_pitch_row, long long rgb_pitch_img,
                       float fx, float fy, float cx, float cy, int u0, int v0, const float* T_host, float trunc,
                       float max_weight, float max_depth, void* stream);
int dca_tsdf_count_surface(const float* volume, int planes, int nx, int ny, int nz, float min_weight,
                           long long* workspace, long long* count, void* stream);
int dca_tsdf_extract_surface(const float* volume, int planes, int nx, int ny, int nz, float ox, float oy, float oz,
                             float voxel_size, float min_weight, const long long* workspace, long long capacity,
                             float* xyz, float* normal, unsigned char* rgb, void* stream);

/* (13) camera tracking against the fused volume: raycast model maps and projective point-to-plane ICP ------------ */
/* The tracking half of KinectFusion (Newcombe et al., ISMAR 2011) with the linearised point-to-plane system of Low (2004).
 * fp32 steps use the notation of section 12 ((+) (-) (x) (/) correctly rounded, no contraction, matrix rows applied as
 * ((m0 a (+) m1 b) (+) m2 c) (+) m3); fp64 steps are __dadd_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn, a - b as
 * a + (-b).  Window pixel (x, y) is image pixel (x + u0, y + v0), as in dca_reproject and dca_tsdf_integrate.
 *
 * dca_tsdf_raycast.  Renders a volume in the state layout of section 12 through an H x W pinhole window.  M = T_host, the
 * camera-to-world 3x4 (row-major, a HOST pointer that travels as launch parameters).  Per pixel:
 *   xn = ((fp32(x) (+) fp32(u0)) (-) cx) (/) fx,  yn = ((fp32(y) (+) fp32(v0)) (-) cy) (/) fy
 *   L = sqrt((xn (x) xn (+) yn (x) yn) (+) 1)           (ray length per metre of camera Z)
 *   the sample at camera Z = z: c = (xn (x) z, yn (x) z, z), p = M c, g = ((p_a (-) o_a) (/) vs) per axis (grid units,
 *       voxel centres at integers); it is UNKNOWN when a corner of its cell (floorf(g), floorf(g) + 1 per axis) lies
 *       outside the grid or has weight < min_weight, else T = trilinear tsdf:
 *       lerp(a, b, t) = a (+) t (x) (b (-) a) along x (fraction g_x (-) floorf(g_x)), then y, then z
 *   march: z = min_depth, no previous sample; while z <= max_depth:
 *       known T:  if the previous sample is known with Tp >= 0 and T < 0: hit, zh = zp (+) (z (-) zp) (x) (Tp (/) (Tp (-) T)),
 *                 stop;  if the previous sample is known with Tp < 0 and T >= 0 (the back of a surface): stop, no hit;
 *                 else s = max(vs (x) 0.5, |T| (x) trunc)
 *       unknown:  s = trunc, and the next sample has no known previous sample (unknown samples never end the march)
 *       z' = z (+) (s (/) L); stop (no hit) unless z' > z;  z = z'
 *   Every step is at most trunc of ray length (|T| <= 1), so a known band of trunc on each side of a surface, crossed by
 *   the ray over at least trunc of its length per band, holds a sample on each side: the ray cannot step over it.
 *   With a hit at zh > 0, at h = the sample point of zh (c, p and g as above):
 *     gradient  G_a = C(g (+) e_a) (-) C(g (-) e_a) per axis, C = the clamped trilinear tsdf: each coordinate clamped
 *               into [0, n - 1], cell corner min(floorf, n - 2), weights ignored; len = sqrt((Gx Gx (+) Gy Gy) (+) Gz Gz);
 *               len = 0 is no hit.  n_world = G (/) len (pointing from behind the surface towards the camera)
 *     outputs   depth = zh (camera Z, the convention of dca_reproject's depth map);  vertex = (xn (x) zh, yn (x) zh, zh)
 *               in the camera frame;  normal_k = ((M0k nwx (+) M1k nwy) (+) M2k nwz) (M^T n_world: camera frame);
 *               rgb_c = clamp(rint(C_c(g)), 0, 255) (round half to even) with C_c the clamped trilinear colour plane
 *   No hit: depth 0, vertex and normal NaN, rgb (0, 0, 0).
 * Outputs fp32 depth [H][depth_pitch], vertex [H][vertex_pitch] (x, y, z per pixel), normal [H][normal_pitch], uint8
 * rgb [H][rgb_pitch] (NULL = not written; planes = 5 only); pitches in elements (bytes for rgb).  One launch, no host
 * sync, no allocation.  DCA_ERR_ARG for NULL volume / T_host / depth / vertex / normal, planes other than 2 or 5, nx, ny
 * or nz < 2, non-finite origin, voxel_size not > 0, trunc not finite and > 0, a NaN min_weight, non-finite or zero
 * fx / fy, non-finite cx / cy, min_depth not >= 0, max_depth not finite or < min_depth, a non-finite T_host, H, W <= 0,
 * depth_pitch < W, vertex_pitch or normal_pitch < 3 W, rgb with planes = 2 or rgb_pitch < 3 W; DCA_ERR_UNSUPPORTED for
 * N >= 2^31, H W >= 2^31, H, W, nx, ny or nz >= 2^24 and |u0| or |v0| >= 2^24.
 *
 * dca_icp_track.  All ICP iterations of one frame.  The source is a depth map (weight optional) of the window, element
 * (y, x) at y pitch + x; the model is the vertex and normal maps of dca_tsdf_raycast with the same intrinsics and window,
 * in the model camera's frame (pitches in elements).  A = T(model camera <- current camera), fp64 3x4, starts at A0_host
 * (a HOST pointer that travels as launch parameters).  Levels l = 0..num_levels-1 run level_iters[l] iterations each
 * with pixel stride s = level_stride[l] and distance gate G = level_gate[l] (fp32).  Per iteration, with Af = fp32(A)
 * (rounded once), for each source pixel (x, y) with x % s = y % s = 0:
 *   z = depth;  keep only z finite and 0 < z <= max_depth
 *   w = 1 without weight, else the weight clamped to [0, 1], 0 where NaN;  keep only w > 0
 *   p = ((((fp32(x) (+) fp32(u0)) (-) cx) (x) z) (/) fx, (((fp32(y) (+) fp32(v0)) (-) cy) (x) z) (/) fy, z)
 *   q = Af p;  keep only 0 < q_z <= Q, |q_x| <= Q, |q_y| <= Q with Q = 2 (x) max_depth
 *   xm = floorf((((fx (x) q_x) (/) q_z) (+) cx) (-) fp32(u0) (+) 0.5), ym likewise; keep only 0 <= xm < W, 0 <= ym < H
 *   m, n = model vertex and normal at (xm, ym);  keep only (n.n) <= DCA_ICP_MAX_NORMAL2 (false for NaN: no model hit)
 *   d = q (-) m;  keep only (dx dx (+) dy dy) (+) dz dz <= G (x) G (false for NaN)
 *   r = (nx dx (+) ny dy) (+) nz dz;  J = (q x n, n) with (q x n) = (qy nz (-) qz ny, qz nx (-) qx nz, qx ny (-) qy nx):
 *       the Jacobian of r for the left-multiplied update (omega, t)
 *   sums, each term rounded to an integer (round half to even) after an exact scaling by a power of two:
 *       H_ij (i <= j, row-major upper triangle) += rint(((w (x) J_i) (x) J_j) * DCA_ICP_SCALE_H)
 *       g_i += rint(((w (x) J_i) (x) r) * DCA_ICP_SCALE_G);  e += rint(((w (x) r) (x) r) * DCA_ICP_SCALE_E)
 *       sw += rint(w * DCA_ICP_SCALE_W);  count += 1
 *   Integer sums are exact and order-free: each CTA of DCA_ICP_TILE pixels of the stride grid writes its int64 row to
 *   the workspace, and one CTA adds the rows.  No sum overflows while max_depth <= DCA_ICP_MAX_DEPTH, G <=
 *   DCA_ICP_MAX_GATE and H W <= DCA_ICP_MAX_PIXELS: |J_i| <= |q||n| <= 2 sqrt(3) max_depth 1.031 < 4 max_depth <= 2^10,
 *   |r| <= 1.031 G (1 + 2^-20) <= 2^4 1.04, so a term is below 2^38 (1.09) of its unit and H W of them below 2^63.  There is
 *   no normal-compatibility test on the source side: stereo normals from forward differences are much noisier than the
 *   raycast normals, and the gate, the confidence weight and the left-right filter already applied by dca_reproject
 *   reject the outliers such a test would.
 *   solve (fp64, one thread): H, g, e, sw = the int64 sums converted to fp64 (correctly rounded) times the inverse
 *       scales;  fail with DCA_ICP_FEW_INLIERS when count < min_inliers;  Cholesky H = L L^T, column j = 0..5:
 *       s = H_jj - L_j0 L_j0 - ... - L_j,j-1 L_j,j-1 (left to right); fail with DCA_ICP_DEGENERATE unless
 *       s > DCA_ICP_PIVOT_REL (x) max_i H_ii;  L_jj = sqrt(s);  L_ij = (H_ij - L_i0 L_j0 - ... ) / L_jj for i > j;
 *       forward  y_i = (-g_i - L_i0 y_0 - ... - L_i,i-1 y_i-1) / L_ii;  backward xi_i = (y_i - L_i+1,i xi_i+1 - ... -
 *       L_5i xi_5) / L_ii  (k ascending);  (omega, t) = xi
 *   update: (hx, hy, hz) = omega (x) 0.5, nq = sqrt(((1 + hx hx) + hy hy) + hz hz), (w, x, y, z) = (1, hx, hy, hz) / nq;
 *       R = [[1 - 2 (yy + zz), 2 (xy - wz), 2 (xz + wy)], [2 (xy + wz), 1 - 2 (xx + zz), 2 (yz - wx)],
 *            [2 (xz - wy), 2 (yz + wx), 1 - 2 (xx + yy)]] (each product and sum rounded as written);
 *       A <- [R | t] A: A'_ij = ((R_i0 A_0j + R_i1 A_1j) + R_i2 A_2j) (+ t_i for j = 3).  A failed iteration leaves A.
 * Outputs (device): pose fp64 [12] = the final A; stats fp64 [total iterations][4] = (count, sw, e, flag) per
 * iteration, flag 0 or DCA_ICP_FEW_INLIERS or DCA_ICP_DEGENERATE; ok int32 = 1 when no iteration failed, else 0.
 * workspace = DCA_ICP_WORKSPACE_BYTES(H, W) bytes.  Fixed iteration counts (no early exit): 2 launches per iteration,
 * no host sync, no allocation: capturable in a CUDA graph.  DCA_ERR_ARG for NULL depth / model maps / A0_host / level
 * arrays / workspace / pose / stats / ok, H, W <= 0, pitch < W, vertex_pitch or normal_pitch < 3 W, non-finite or zero
 * fx / fy, non-finite cx / cy, max_depth not finite and > 0, min_inliers < 1, num_levels outside
 * 1..DCA_ICP_MAX_LEVELS, a stride < 1, iterations outside 1..DCA_ICP_MAX_ITERS, a gate not finite and > 0 and a
 * non-finite A0; DCA_ERR_UNSUPPORTED for max_depth > DCA_ICP_MAX_DEPTH, a gate > DCA_ICP_MAX_GATE, H W >
 * DCA_ICP_MAX_PIXELS and |u0| or |v0| >= 2^24. */
#define DCA_ICP_TILE 1024
#define DCA_ICP_WORKSPACE_ROW 32
#define DCA_ICP_WORKSPACE_BYTES(H, W)                                                                                 \
  (8ull * DCA_ICP_WORKSPACE_ROW *                                                                                     \
   (((unsigned long long)(H) * (unsigned long long)(W) + DCA_ICP_TILE - 1) / DCA_ICP_TILE))
#define DCA_ICP_MAX_LEVELS 4
#define DCA_ICP_MAX_ITERS 64
#define DCA_ICP_MAX_DEPTH 256.0f
#define DCA_ICP_MAX_GATE 16.0f
#define DCA_ICP_MAX_PIXELS (1ll << 24)
#define DCA_ICP_MAX_NORMAL2 1.0625f
#define DCA_ICP_SCALE_H 262144.0f      /* 2^18 */
#define DCA_ICP_SCALE_G 16777216.0f    /* 2^24 */
#define DCA_ICP_SCALE_E 1073741824.0f  /* 2^30 */
#define DCA_ICP_SCALE_W 1073741824.0f  /* 2^30 */
#define DCA_ICP_PIVOT_REL 5e-5        /* DESIGN.md, "Tracking": between a ground plane (<= 1.3e-5) and the full scene (>= 3e-4) */
#define DCA_ICP_FEW_INLIERS 1
#define DCA_ICP_DEGENERATE 2
int dca_tsdf_raycast(const float* volume, int planes, int nx, int ny, int nz, float ox, float oy, float oz,
                     float voxel_size, float trunc, float min_weight, float fx, float fy, float cx, float cy, int u0,
                     int v0, int H, int W, const float* T_host, float min_depth, float max_depth, float* depth,
                     long long depth_pitch, float* vertex, long long vertex_pitch, float* normal,
                     long long normal_pitch, unsigned char* rgb, long long rgb_pitch, void* stream);
int dca_icp_track(const float* depth, const float* weight, long long pitch, int H, int W, float fx, float fy, float cx,
                  float cy, int u0, int v0, float max_depth, const float* model_vertex, long long vertex_pitch,
                  const float* model_normal, long long normal_pitch, const double* A0_host, int num_levels,
                  const int* level_stride, const int* level_iters, const float* level_gate, int min_inliers,
                  void* workspace, double* pose, double* stats, int* ok, void* stream);

/* layout + parameter preparation ---------------------------------------------------------------- */
int dca_planes_from_ncdhw(const float* x, void* y, int planes, int B, int C, int Cp, int D, int H, int W,
                          void* stream);
int dca_planes_to_ncdhw(const void* x, int planes, float* y, int B, int C, int Cp, int D, int H, int W, void* stream);
/* cost planes [planes][B][1][H][W][Cp] -> a C-channel slice of a wider fp32 NCHW tensor (batch pitch y_batch_stride
 * elements): torch.cat((l2, l3, l4), dim=1) of feature_extraction.forward (gwcnet_dca_g.py:60) without the copy. */
int dca_planes_to_nchw_slice(const void* x, int planes, float* y, int B, int C, int Cp, int H, int W,
                             long long y_batch_stride, void* stream);
int dca_pack_weights(const float* w, int transposed, int Co, int Ci, int taps, float* out, int CoPad, void* stream);
int dca_fold_bn(const float* gamma, const float* beta, const float* mean, const float* var, float eps, float* scale,
                float* shift, int C, int Cpad, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DCA_B200_H */
