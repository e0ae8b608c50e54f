/*
 * damvs.h -- C ABI of the B200-native DA-MVSNet cost-volume hot path.
 *
 * One shared library (damvsnet_b200/_C/libdamvs_b200.so, sm_100a only).  Plain
 * pointers and sizes, no torch types.  Every pointer marked "device" is a CUDA
 * device pointer the caller owns for the duration of the call; the library never
 * allocates, frees or retains device memory.  Every entry point is asynchronous
 * on `stream` (a cudaStream_t passed as void*), performs no host synchronisation,
 * returns 0 on success and a non-zero code otherwise (never throws, never exits);
 * damvs_last_error() returns the message of the calling thread's last failure.
 *
 * The reference is pure Python (no FFI of its own), so each entry point cites the
 * reference Python function whose arithmetic it replaces; INTEGRATION.md shows
 * the ctypes binding a maintainer would add to the reference.
 *
 * Activation layout ("G8"): a logical [B,C,D,H,W] volume is stored as
 * [B][C/8][D][H][W][8] -- eight channels innermost (16 B in bf16, 32 B in fp32),
 * channel groups outermost, so that every 8-channel group is a dense D*H*W
 * volume that TMA can tile with a contiguous inner dimension of W*8 elements.
 * Feature maps are NHWC fp32: [B][H][W][C].
 */
#ifndef DAMVS_H_
#define DAMVS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAMVS_ABI_VERSION 1

enum damvs_status {
  DAMVS_OK = 0,
  DAMVS_ERR_INVALID = 1,     /* bad argument (shape, dtype, alignment, null) */
  DAMVS_ERR_UNSUPPORTED = 2, /* valid request this build has no kernel for */
  DAMVS_ERR_CUDA = 3,        /* CUDA runtime/driver error (message has cudaGetErrorString) */
  DAMVS_ERR_NO_DEVICE = 4    /* device is not sm_100 */
};

/* Element types of cost volumes / CostRegNet activations.  DAMVS_F16 (IEEE half: 11 significand bits, 8x finer than
 * bf16 at the same width and the same tensor-core rate) is the inference pipeline's reduced-precision format; values
 * saturate to +-65504 on store.  DAMVS_BF16 stays the training format (gradients need the exponent range). */
enum damvs_dtype { DAMVS_F32 = 0, DAMVS_BF16 = 1, DAMVS_F16 = 2 };
enum damvs_agg_mode { DAMVS_AGG_VARIANCE = 0, DAMVS_AGG_ADAPTIVE = 1 };
enum damvs_conv_impl { DAMVS_CONV_DIRECT = 0, DAMVS_CONV_TCGEN05 = 1 };

int damvs_abi_version(void);
const char* damvs_last_error(void);
/* 0 when device `dev` can run this library (compute capability 10.x). */
int damvs_check_device(int dev);

/* ---- layout helpers ----------------------------------------------------- */
/* [B,C,H,W] fp32 -> [B,H,W,C] fp32.  Feature maps handed over in the reference's
 * NCHW layout (models/cas_mvsnet.py:24 `features`) are repacked once per view. */
int damvs_nchw_to_nhwc_f32(const float* in, float* out, int B, int C, int H, int W, void* stream);
/* [B,C,D,H,W] fp32 <-> G8 volume of `dtype`.  C % 8 == 0. */
int damvs_ncdhw_to_g8(const float* in, void* out, int dtype, int B, int C, int D, int H, int W, void* stream);
int damvs_g8_to_ncdhw(const void* in, int dtype, float* out, int B, int C, int D, int H, int W, void* stream);

/* ---- homography warp (stand-alone) --------------------------------------- */
/* Replaces homo_warping (reference models/module.py:297-332) from the sampling
 * grid onwards; `rot_trans` holds, per batch item, rows 0-2 of
 * src_proj @ inverse(ref_proj) as 12 floats (rot row-major, then trans), computed
 * by the caller exactly as models/module.py:308-310 does.
 *   src_nhwc   device [B,H,W,C] fp32
 *   rot_trans  device [B,12] fp32
 *   depth_hyp  device [B,D,H,W] (per_pixel_hyp=1) or [B,D] (per_pixel_hyp=0) fp32
 *   out        device [B,C,D,H,W] fp32 (the reference's output layout)            */
int damvs_homo_warp_fwd(const float* src_nhwc, const float* rot_trans, const float* depth_hyp, float* out,
                        int B, int C, int D, int H, int W, int per_pixel_hyp, void* stream);

/* ---- fused warp + multi-view aggregation --------------------------------- */
/* Replaces the source-view loop of DepthNet.forward (reference
 * models/cas_mvsnet.py:30-87): ref-volume repeat, homo_warping per source view,
 * variance or adaptive aggregation including AggWeightNetVolume in eval mode
 * (models/module.py:544-563).  The N x D warped volume never reaches memory.
 *   ref_nhwc    device [B,H,W,C] fp32
 *   src_nhwc    HOST array of n_src device pointers, each [B,H,W,C] fp32
 *   rot_trans   device [n_src,B,12] fp32 (see damvs_homo_warp_fwd)
 *   depth_hyp   device [B,D,H,W] or [B,D] fp32
 *   wnet        device [C+5] fp32: w1[C], scale1, shift1, w2, scale2, shift2 -- the
 *               two 1x1x1 convs of w_net and their folded eval-mode BatchNorms;
 *               NULL for DAMVS_AGG_VARIANCE
 *   out_vol     device G8 volume [B,C/8,D,H,W,8] of out_dtype
 * C in {8,16,32,64}; n_src in [1,15].                                            */
int damvs_warp_agg_fwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                       const float* depth_hyp, const float* wnet, void* out_vol, int B, int C, int D, int H,
                       int W, int mode, int per_pixel_hyp, int out_dtype, void* stream);

/* ---- 3-D convolution blocks of CostRegNet -------------------------------- */
/* One Conv3d / Deconv3d block of the reference (models/module.py:117-202) with
 * eval-mode BatchNorm folded to a per-channel affine, optional ReLU, and the
 * additive U-Net skip of CostRegNet.forward (models/module.py:532-541) fused:
 *     out = skip + act(conv(in) * scale + shift)
 * kernel 3x3x3, padding 1; stride 1 or 2; transposed => ConvTranspose3d(k3, s2,
 * p1, output_padding 1) whose output extent is twice the input's.               */
typedef struct damvs_conv3d_desc {
  int B, Cin, Cout;        /* Cin % 8 == 0; Cout % 8 == 0, or Cout == 1 with plain_out */
  int Din, Hin, Win;       /* input extent */
  int stride;              /* 1 or 2 (ignored when transposed) */
  int transposed;          /* 0: Conv3d, 1: ConvTranspose3d(k3,s2,p1,op1) */
  int relu;                /* apply ReLU after the affine */
  int in_dtype, out_dtype; /* damvs_dtype of the G8 input / output volumes */
  int plain_out;           /* 1: Cout == 1, output is plain fp32 [B,D,H,W] (the `prob` conv) */
  int impl;                /* damvs_conv_impl */
} damvs_conv3d_desc;

/* Bytes of the packed weight buffer for (desc->impl, Cin, Cout). */
size_t damvs_conv3d_packed_weight_bytes(const damvs_conv3d_desc* desc);
/* Repack a PyTorch-layout fp32 weight (Conv3d: [Cout,Cin,3,3,3]; ConvTranspose3d:
 * [Cin,Cout,3,3,3]; device pointer) into the layout `impl` consumes. */
int damvs_conv3d_pack_weight(const damvs_conv3d_desc* desc, const float* weight, void* packed, void* stream);
/*   in      device G8 volume [B,Cin/8,Din,Hin,Win,8]
 *   packed  device, from damvs_conv3d_pack_weight
 *   scale, shift  device [Cout] fp32, or NULL for identity (the `prob` conv has no BN)
 *   skip    device, same layout/dtype as out, or NULL
 *   out     device G8 volume of the output extent, or plain fp32 when plain_out  */
int damvs_conv3d_fwd(const damvs_conv3d_desc* desc, const void* in, const void* packed, const float* scale,
                     const float* shift, const void* skip, void* out, void* stream);

/* ---- half-precision feature path (the bf16 pipeline's producer) ---------------
 * Same operation as damvs_nchw_to_nhwc_f32 / damvs_warp_agg_fwd with the feature maps held as fp16 NHWC
 * (values saturate at +-65504): half the gather traffic, fp32 accumulation in the blend, coordinates equal to
 * the reference's up to fp32 rounding instead of bit-exact.  Used when the cost volume is emitted in bf16.   */
int damvs_nchw_to_nhwc_f16(const float* in, void* out, int B, int C, int H, int W, void* stream);
/* n (<= 16) equally shaped feature maps in one launch; ins / outs are HOST arrays of device pointers. */
int damvs_nchw_to_nhwc_f16_multi(const float* const* ins, void* const* outs, int n, int B, int C, int H, int W, void* stream);
int damvs_warp_agg_fwd_f16(const void* ref_nhwc, const void* const* src_nhwc, int n_src, const float* rot_trans,
                           const float* depth_hyp, const float* wnet, void* out_vol, int B, int C, int D, int H,
                           int W, int mode, int per_pixel_hyp, int out_dtype, void* stream);

/* ---- group-wise correlation aggregation (NOT in the reference) ----------------
 * The third aggregation mode BASELINE.json's north star names (configs[4], "groups 4-32"); the reference has only
 * variance / adaptive (models/cas_mvsnet.py:14, 34-39).  cost[g] = mean over source views of the mean over the C/G
 * channels of group g of ref * warp, with the reference's homography warp (models/module.py:297-332).
 *   ref_nhwc, src_nhwc[v]  NHWC features, fp32 or fp16 (feat_dtype = DAMVS_F32 | DAMVS_F16)
 *   out_vol                G8 volume of max(G, 8) channels (G = 4: channels 4..7 are written as zero), out_dtype any
 *   C in {8,16,32}, G in {4,8,16,32}, G <= C.  Other arguments as damvs_warp_agg_fwd.                              */
int damvs_warp_gwc_fwd(const void* ref_nhwc, const void* const* src_nhwc, int n_src, const float* rot_trans,
                       const float* depth_hyp, void* out_vol, int B, int C, int G, int D, int H, int W,
                       int per_pixel_hyp, int feat_dtype, int out_dtype, void* stream);

/* ---- group-wise correlation, training forward and backward ---------------------------------------------------
 * The forward and the backward sample at bit-identical coordinates (the reference's operation order, as the other
 * training kernels), so the gradient is that of the volume the forward returned.  S = C/G, k = 1/(n_src S):
 *   fwd: out_vol[g] = k sum_v sum_{c in g} ref[c] warp_v[c]; fp32 NHWC features, G8 volume of max(G, 8) channels in
 *        out_dtype = DAMVS_F32 | DAMVS_BF16 (G = 4: channels 4..7 written as zero).
 *   bwd: g_vol (G8, g_dtype = DAMVS_F32 | DAMVS_BF16; padding channels of G = 4 are ignored) ->
 *        g_ref[c] = k sum_d g_vol[g(c)] sum_v warp_v[c]  (overwritten),
 *        g_src[v] += bilinear scatter of k g_vol[g(c)] ref[c]  (ACCUMULATED with vector atomics: zero them first;
 *        HOST array of device pointers).  The sampling grid and the hypotheses receive no gradient.
 * C in {8,16,32}, G in {4,8,16,32}, G <= C, n_src in [1,15].  Other arguments as damvs_warp_agg_fwd.             */
int damvs_warp_gwc_train_fwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                             const float* depth_hyp, void* out_vol, int B, int C, int G, int D, int H, int W,
                             int per_pixel_hyp, int out_dtype, void* stream);
int damvs_warp_gwc_bwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                       const float* depth_hyp, const void* g_vol, int g_dtype, float* g_ref, float* const* g_src, int B,
                       int C, int G, int D, int H, int W, int per_pixel_hyp, void* stream);

/* ---- fused `prob` convolution + head ------------------------------------------
 * CostRegNet's last layer (models/module.py:530: Conv3d 8 -> 1, k3, p1, no bias) and the softmax / regression /
 * confidence / variance head (models/cas_mvsnet.py:105-124) in ONE launch: the logits stay in shared memory.
 * desc as for damvs_conv3d_fwd with plain_out = 1, impl = DAMVS_CONV_TCGEN05; packed = the same blob damvs_conv3d_fwd
 * takes for that layer.  depth_hyp, prob: device fp32 [B][D][H][W]; depth, conf, var: device fp32 [B][H][W].
 * damvs_prob_head_supported(desc) != 0 iff the shape qualifies (bf16 / fp16 volume, D % 8 == 0, D <= 64); otherwise
 * call damvs_conv3d_fwd + damvs_softmax_regress_fwd.                                                              */
int damvs_prob_head_supported(const damvs_conv3d_desc* desc);
int damvs_prob_head_fwd(const damvs_conv3d_desc* desc, const void* in, const void* packed, const float* depth_hyp,
                        float* prob, float* depth, float* conf, float* var, void* stream);

/* ---- softmax / regression head -------------------------------------------- */
/* Replaces models/cas_mvsnet.py:105-124 + depth_regression (models/module.py:609):
 * softmax over D, expected depth, photometric confidence (sum of p over
 * [idx-1, idx+2] at idx = trunc(sum p*k)), and 3*sqrt(sum p (d - depth)^2).
 *   logits     device [B,D,H,W] fp32
 *   depth_hyp  device [B,D,H,W] or [B,D] fp32
 *   prob       device [B,D,H,W] fp32 out (may be NULL to skip the store)
 *   depth, conf, var   device [B,H,W] fp32 out                                   */
int damvs_softmax_regress_fwd(const float* logits, const float* depth_hyp, float* prob, float* depth,
                              float* conf, float* var, int B, int D, int H, int W, int per_pixel_hyp,
                              void* stream);
/* depth_regression alone (models/module.py:609-615): out[b,h,w] = sum_d p * d. */
int damvs_depth_regression_fwd(const float* prob, const float* depth_hyp, float* out, int B, int D, int H,
                               int W, int per_pixel_hyp, void* stream);

/* ---- backward ----------------------------------------------------------------- */
/* The reference's backward is PyTorch autograd; these are the native counterparts for the hot path.
 * Data gradients of a conv block are one more damvs_conv3d_fwd call with re-packed weights (the adjoint of a
 * stride-1 conv is a stride-1 conv with transposed + flipped weights, of a stride-2 conv the transposed
 * conv, and vice versa) -- see damvsnet_b200/autograd.py.                                              */

/* Gradient of the head (models/cas_mvsnet.py:105-124) w.r.t. the logits:
 *   g_logit[k] = p_k (g_p[k] - sum_j p_j g_p[j]),  g_p[k] = g_depth d_k + g_var 3/(2 sqrt S) (d_k - depth)^2 + g_prob[k]
 * g_depth, g_var, g_prob: incoming gradients, any may be NULL (= zero).  g_hyp (optional, per-pixel hypotheses
 * only) receives d/d depth_values for grad_method "undetach".  photometric_confidence has no gradient
 * (computed under no_grad in the reference, cas_mvsnet.py:113).                                           */
int damvs_softmax_regress_bwd(const float* prob, const float* depth_hyp, const float* depth, const float* g_depth,
                              const float* g_var, const float* g_prob, float* g_logits, float* g_hyp, int B, int D,
                              int H, int W, int per_pixel_hyp, void* stream);

/* ---- training-mode BatchNorm3d around the conv blocks (models/module.py:141-159, 184-202) ---------------
 * In training the conv kernels write the raw convolution y (damvs_conv3d_fwd with scale = shift = skip = NULL,
 * relu = 0); these three streaming kernels do the rest on G8 volumes of `dtype`.  The C-sized coefficient
 * algebra (statistics -> scale/shift, BatchNorm backward -> k1,k2,k3, running buffers) is the caller's.   */

/* sums[c] += {sum y, sum y^2} over (B,D,H,W); sums is fp64 [C][2], ACCUMULATED (zero it first). */
int damvs_bn_stats(const void* y, int dtype, int B, int C, int D, int H, int W, double* sums, void* stream);

/* out = skip + act(y * scale[c] + shift[c]); skip may be NULL; out may alias y. */
int damvs_bn_apply(const void* y, const float* scale, const float* shift, const void* skip, void* out, int dtype, int B,
                   int C, int D, int H, int W, int relu, void* stream);

/* Backward of damvs_bn_apply.  g_z = g_out * [act active] with the activation recomputed from y, scale, shift;
 *   sums[c] += {sum g_z, sum g_z * y}   (fp64 [C][2], ACCUMULATED; NULL to skip)
 *   g_y = k1[c] * g_z + k2[c] * y + k3[c]  (NULL k1 = 1, NULL k2/k3 = 0; g_y NULL to skip)
 * Batch statistics need two calls (sums, then g_y with the BatchNorm-backward coefficients); fixed statistics
 * one call with k1 = scale.  The gradient of the skip input is g_out itself.                              */
int damvs_bn_bwd(const void* g_out, const void* y, const float* scale, const float* shift, const float* k1, const float* k2,
                 const float* k3, void* g_y, double* sums, int dtype, int B, int C, int D, int H, int W, int relu,
                 void* stream);

/* The C-sized coefficient algebra between those kernels, one launch each (device pointers, [C] fp32 unless noted).
 * finalize: sums (fp64 [C][2] from damvs_bn_stats over `count` voxels) -> batch mean / rstd, scale = gamma * rstd,
 *   shift = beta - mean * scale; running_mean / running_var (NULL to skip) are updated in place with `momentum` and
 *   the unbiased variance, as nn.BatchNorm3d.forward does in training.
 * bwd_coeffs: sums (fp64 [C][2] from damvs_bn_bwd) -> g_gamma, g_beta and, for batch statistics, k1, k2, k3 of
 *   damvs_bn_bwd's second call (NULL for fixed statistics).                                                     */
int damvs_bn_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                      double count, float momentum, float eps, float* scale, float* shift, float* mean, float* rstd, int C,
                      void* stream);
int damvs_bn_bwd_coeffs(const double* sums, const float* scale, const float* mean, const float* rstd, double count, float* k1,
                        float* k2, float* k3, float* g_gamma, float* g_beta, int C, void* stream);

/* [voxels] fp32 -> G8 volume of one channel group: channel 0 = value, channels 1..7 = 0 (gradient of the
 * single-channel `prob` convolution's output, fed to the adjoint convolution and to damvs_conv3d_wgrad). */
int damvs_plain_to_g8(const float* in, void* out, int dtype, long long voxels, void* stream);

/* Weight gradient of a conv block in PyTorch layout (Conv3d [Cout,Cin,3,3,3], ConvTranspose3d [Cin,Cout,3,3,3]),
 * fp32, overwritten.  desc describes the FORWARD convolution; in_dtype / out_dtype are the dtypes of x and g_y. */
int damvs_conv3d_wgrad(const damvs_conv3d_desc* desc, const void* x, const void* g_y, float* dw, void* stream);

/* Backward of damvs_warp_agg_fwd: g_vol (G8, g_dtype) -> g_ref [B,H,W,C] (overwritten), g_src[v] [B,H,W,C]
 * (ACCUMULATED with vector atomics: zero them first; HOST array of device pointers), g_wnet [C+5] gradients
 * of the folded view-weight parameters in the layout of `wnet` (ACCUMULATED; NULL to skip; adaptive only).
 * The sampling grid and the hypotheses receive no gradient, as in the reference (models/module.py:307).   */
int damvs_warp_agg_bwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                       const float* depth_hyp, const float* wnet, const void* g_vol, int g_dtype, float* g_ref,
                       float* const* g_src, float* g_wnet, int B, int C, int D, int H, int W, int mode,
                       int per_pixel_hyp, void* stream);

/* ---- warp + aggregation with the view-weight net in training mode (batch statistics) --------------------
 * AggWeightNetVolume's BatchNorms (models/module.py:548-551) then normalise over a whole per-view score volume,
 * so the adaptive aggregation splits into  s_v = sum_c w1[c] (ref - warp_v)[c]^2  ("score"),  the scalar
 * chain s_v -> wt_v on [n_src][B][D][H][W] fp32 volumes (damvs_wnet_chain_fwd), and
 * vol = sum_v (wt_v + 1)(ref - warp_v)^2 / n_src ("weighted").                                                */
int damvs_warp_score_fwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                         const float* depth_hyp, const float* w1, float* s_vol, int B, int C, int D, int H, int W,
                         int per_pixel_hyp, void* stream);
int damvs_warp_weighted_fwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                            const float* depth_hyp, const float* wt_vol, void* out_vol, int B, int C, int D, int H, int W,
                            int per_pixel_hyp, int out_dtype, void* stream);

/* ---- depth-hypothesis sampling for cascade stages 2/3 (upstream neighbour of the path) ----------------
 * Fuses models/cas_mvsnet.py:250-253 (two bilinear up-samples to full resolution), uncertainty_aware_samples
 * (models/module.py:999-1038, the `cur_depth.dim() != 2` branch) and the trilinear resample of
 * models/cas_mvsnet.py:293-296 into one kernel:
 *   prev_depth, prev_var  device [B,hp,wp] fp32: `depth` and `variance` of the previous stage
 *   out                   device [B,D,H/scale,W/scale] fp32: the depth_values DepthNet.forward receives
 * (H,W) is the full image size, scale in {1,2,4} the stage scale.  With hp = H, wp = W, scale = 1 it is
 * uncertainty_aware_samples alone on full-resolution [B,1,H,W] inputs.                                   */
int damvs_uncertainty_samples_fwd(const float* prev_depth, const float* prev_var, float* out, int B, int hp, int wp, int D,
                                  int H, int W, int scale, void* stream);

/* ---- geometric-consistency filtering of one reference view (downstream neighbour of the path) ----------
 * Fuses reproject_with_depth + check_geometric_consistency (filter/dypcd.py:98-159) and the accumulation over
 * the source views of filter_depth (filter/dypcd.py:205-257) into one kernel.
 *   depth_ref, conf1..3  device [H,W] fp32: the reference view's depth and its stage-1/2/3 confidence maps
 *   depth_src            HOST array of n_src device pointers, [H,W] fp32 each
 *   cams                 HOST float64: K_ref[9], inv(K_ref)[9], then per source view 42 values:
 *                        (E_src inv(E_ref)) rows 0-2 [12], K_src [9], inv(K_src) [9], (E_ref inv(E_src)) rows 0-2 [12]
 *   conf_thr1..3         photometric thresholds (args.conf), dist_base / rel_diff_base the dynamic-consistency bases
 *   depth_avg [H,W] fp32, photo_mask / geo_mask / final_mask [H,W] uint8 out;  n_src <= 10                     */
int damvs_geo_consistency_fuse(const float* depth_ref, const float* conf1, const float* conf2, const float* conf3,
                               const float* const* depth_src, const double* cams, int n_src, int H, int W,
                               float conf_thr1, float conf_thr2, float conf_thr3, double dist_base, double rel_diff_base,
                               float* depth_avg, uint8_t* photo_mask, uint8_t* geo_mask, uint8_t* final_mask, void* stream);

/* ---- cross-view photometric loss (training-side neighbour of the path) -----------------------------------
 * Fuses cross_view_loss (models/module.py:624-691) and inverse_warping (models/homography.py:7-201) for one stage:
 *   depth_est, depth_gt  device [B,H,W] fp32
 *   view_imgs            HOST array of n_src device pointers, [B,3,H,W] fp32 (source images at the stage resolution)
 *   cams                 device [B][n_src][21] fp32: inv(K_ref) [9], rows 0-2 of [K_ref|0;0001][R_rel|t_rel;0001] [12]
 * terms:  maskbits [B,H,W] uint16 out (bit v: both warps of source view v valid), sums[v] += smooth-L1 sum (fp64,
 *         ACCUMULATED; L_v = sums[v] / (B*H*W*3)).
 * select: counts[v] += number of pixels that pick view v among their two smallest valid L_v (ACCUMULATED).
 * bwd:    g_depth [B,H,W] out = sum_v coeff[v] * d(smooth-L1 sum of view v)/d depth_est  (coeff: device [n_src]).   */
int damvs_cross_view_terms(const float* depth_est, const float* depth_gt, const float* const* view_imgs, const float* cams,
                           int B, int n_src, int H, int W, uint16_t* maskbits, double* sums, void* stream);
int damvs_cross_view_select(const uint16_t* maskbits, const float* losses, int n_src, long long npix,
                            unsigned long long* counts, void* stream);
int damvs_cross_view_bwd(const float* depth_est, const float* depth_gt, const float* const* view_imgs, const float* cams,
                         const float* coeff, int B, int n_src, int H, int W, float* g_depth, void* stream);

/* The scalar chain between them, s_v -> wt_v = relu(bn2(w2 relu(bn1(s_v)))) with batch statistics per view (n_src
 * successive calls of the net in the reference), on [n_src][M] fp32 volumes (M = B*D*H*W); all pointers device.
 * fwd: sums_ws fp64 [4*n_src] zeroed by the caller; state fp32 [n_src][8] out (per view: a1, c1, mean1, rstd1, a2, c2,
 *      mean2, rstd2: the folded affines and what the backward needs); running buffers (NULL to skip) updated view by view.
 * bwd: sums_ws fp64 [4*n_src + 2] zeroed; coef_ws fp32 [n_src][6] scratch; g_s [n_src][M] out;
 *      g_params [5] out = d gamma1, d beta1, d w2, d gamma2, d beta2 (summed over views).                            */
int damvs_wnet_chain_fwd(const float* s_vol, int n_src, long long M, const float* gamma1, const float* beta1, float* running_mean1,
                         float* running_var1, const float* w2, const float* gamma2, const float* beta2, float* running_mean2,
                         float* running_var2, float momentum, float eps, double* sums_ws, float* state, float* wt_vol, void* stream);
int damvs_wnet_chain_bwd(const float* s_vol, const float* g_wt, int n_src, long long M, const float* state, const float* w2, double* sums_ws,
                         float* coef_ws, float* g_s, float* g_params, void* stream);

/* The backward of the pair in two passes instead of two scatters: damvs_warp_gwt writes only d loss / d wt_v (no
 * feature gradients); after the caller has pushed it through the scalar chain to d loss / d s_v, damvs_warp_merged_bwd
 * scatters both contributions to the features at once (g_ref, g_src, g_w1 ACCUMULATED).                          */
int damvs_warp_gwt(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans, const float* depth_hyp,
                   const void* g_vol, int g_dtype, float* g_wt_vol, int B, int C, int D, int H, int W, int per_pixel_hyp, void* stream);
int damvs_warp_merged_bwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                          const float* depth_hyp, const float* w1, const float* wt_vol, const float* g_s_vol, const void* g_vol,
                          int g_dtype, float* g_ref, float* const* g_src, float* g_w1, int B, int C, int D, int H, int W,
                          int per_pixel_hyp, void* stream);

/* Number of kernel launches this library has issued in this process (for bench.py's gpu_launches). */
uint64_t damvs_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DAMVS_H_ */
