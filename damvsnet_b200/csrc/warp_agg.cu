// Fused homography warp + multi-view aggregation (forward).
//
// Replaces the source-view loop of DepthNet.forward (reference
// models/cas_mvsnet.py:30-87) together with homo_warping
// (models/module.py:297-332) and AggWeightNetVolume in eval mode
// (models/module.py:544-563).  The reference materialises, per source view, a
// sampling grid, a warped [B,C,D,h,w] volume, its squared difference to a
// repeated reference volume and a weight volume; here each depth plane's
// projection is built in registers, the four bilinear taps are gathered from the
// NHWC source feature map as 16-byte vectors, and the aggregate is accumulated
// on the fly, so the only HBM traffic is the feature maps (read, mostly through
// L2), the hypotheses (read once) and the cost volume (written once, G8 layout,
// optionally bf16).
//
// Algorithmic bytes per launch: N*C*h*w*4 + D*h*w*4 read, C*D*h*w*sizeof(out) written.
//
// Mapping: a thread owns (pixel, 4 consecutive channels) and walks the D
// hypotheses of its pixel; the C/4 lanes of a pixel are adjacent in the warp, so
// one tap of one pixel is a single contiguous C*4-byte segment (a full 128-byte
// line for C=32) and the channel reduction of the view-weight net is a
// log2(C/4)-step xor shuffle.  A warp covers 32/(C/4) consecutive pixels of a
// row, a 256-thread CTA a (2*that) x 4 pixel patch, which keeps the source
// footprint of a CTA compact as it slides along the epipolar lines.
//
// Sampling semantics are the reference's, quirk included (SURVEY.md section 0.3):
// the grid is normalised with (W-1)/2 but sampled with align_corners=False, no
// z>0 mask, no epsilon in the perspective divide, zero padding per tap.
#include <cstdlib>

#include "common.cuh"

namespace damvs {

constexpr int kMaxSrc = 15;

struct WarpAggParams {
  const float* ref;
  const float* src[kMaxSrc];
  const float* rot_trans;  // [n_src][B][12]
  const float* hyp;        // [B][D][H][W] or [B][D]
  const float* wnet;       // [C+5] or null
  void* out;               // G8 [B][C/8][D][H][W][8]
  int B, n_src, D, H, W, per_pixel;
};

// source coordinates of reference pixel (x,y) at depth d, exactly in the
// reference's operation order (mul, add, div kept un-contracted)
__device__ __forceinline__ void project(const float* rt, float rx, float ry, float rz, float d, float inv_half_w,
                                        float inv_half_h, float fw, float fh, float& ix, float& iy) {
  float px = __fadd_rn(__fmul_rn(rx, d), rt[9]);
  float py = __fadd_rn(__fmul_rn(ry, d), rt[10]);
  float pz = __fadd_rn(__fmul_rn(rz, d), rt[11]);
  float u = __fdiv_rn(px, pz);
  float v = __fdiv_rn(py, pz);
  // tensor / python-scalar: ATen's CUDA div kernel multiplies by the fp32 reciprocal of a CPU scalar divisor
  float gx = __fadd_rn(__fmul_rn(u, inv_half_w), -1.f);  // models/module.py:323
  float gy = __fadd_rn(__fmul_rn(v, inv_half_h), -1.f);  // models/module.py:324
  // ATen grid_sampler_unnormalize, align_corners=False
  ix = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(gx, 1.f), fw), -1.f), 0.5f);
  iy = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(gy, 1.f), fh), -1.f), 0.5f);
}

// bilinear sample of 4 channels with zero padding per tap (ATen grid_sampler_2d order nw, ne, sw, se)
__device__ __forceinline__ float4 sample4(const float* __restrict__ img, int H, int W, int C, int c0, float ix,
                                          float iy) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  // NaN / far-out-of-range coordinates sample nothing (ATen returns NaN for NaN coordinates; the
  // synthetic inputs keep z != 0, SURVEY.md H1)
  if (!(ix > -1.f && ix < (float)W && iy > -1.f && iy < (float)H)) return acc;
  float fx0 = floorf(ix), fy0 = floorf(iy);
  int x0 = (int)fx0, y0 = (int)fy0;
  float fx1 = fx0 + 1.f, fy1 = fy0 + 1.f;
  float wnw = (fx1 - ix) * (fy1 - iy);
  float wne = (ix - fx0) * (fy1 - iy);
  float wsw = (fx1 - ix) * (iy - fy0);
  float wse = (ix - fx0) * (iy - fy0);
  bool xl = x0 >= 0, xr = x0 + 1 < W, yt = y0 >= 0, yb = y0 + 1 < H;
  const float* p = img + ((long long)y0 * W + x0) * C + c0;
  float4 t;
  if (yt && xl) {
    t = __ldg(reinterpret_cast<const float4*>(p));
    acc.x += t.x * wnw; acc.y += t.y * wnw; acc.z += t.z * wnw; acc.w += t.w * wnw;
  }
  if (yt && xr) {
    t = __ldg(reinterpret_cast<const float4*>(p + C));
    acc.x += t.x * wne; acc.y += t.y * wne; acc.z += t.z * wne; acc.w += t.w * wne;
  }
  if (yb && xl) {
    t = __ldg(reinterpret_cast<const float4*>(p + (long long)W * C));
    acc.x += t.x * wsw; acc.y += t.y * wsw; acc.z += t.z * wsw; acc.w += t.w * wsw;
  }
  if (yb && xr) {
    t = __ldg(reinterpret_cast<const float4*>(p + (long long)W * C + C));
    acc.x += t.x * wse; acc.y += t.y * wse; acc.z += t.z * wse; acc.w += t.w * wse;
  }
  return acc;
}

// One bilinear footprint in "always addressable" form: `off` is the element offset of a 2x2 tap block
// that lies inside the image, and the four weights are ATen's (nw, ne, sw, se) products with the weight
// of every out-of-range tap set to zero and re-assigned to the in-range tap the clamped block maps it to.
struct Footprint {
  float w00, w01, w10, w11;
  int off;
};

__device__ __forceinline__ Footprint make_footprint(float ix, float iy, int H, int W, int C) {
  Footprint f;
  f.w00 = f.w01 = f.w10 = f.w11 = 0.f;
  f.off = 0;
  // NaN / far-out-of-range coordinates sample nothing (ATen returns NaN for NaN coordinates; the
  // synthetic inputs keep z != 0, SURVEY.md H1)
  if (!(ix > -1.f && ix < (float)W && iy > -1.f && iy < (float)H)) return f;
  const float fx0 = floorf(ix), fy0 = floorf(iy);
  const int x0 = (int)fx0, y0 = (int)fy0;
  float wl = (fx0 + 1.f) - ix, wr = ix - fx0;   // weights of columns x0, x0+1
  float wt = (fy0 + 1.f) - iy, wb = iy - fy0;   // weights of rows y0, y0+1
  int xc = x0, yc = y0;
  if (x0 < 0) { xc = 0; wl = wr; wr = 0.f; }                 // only column 0 (the old right tap) is in range
  else if (x0 > W - 2) { xc = W - 2; wr = wl; wl = 0.f; }    // only column W-1 (the old left tap) is in range
  if (y0 < 0) { yc = 0; wt = wb; wb = 0.f; }
  else if (y0 > H - 2) { yc = H - 2; wb = wt; wt = 0.f; }
  f.w00 = wl * wt; f.w01 = wr * wt; f.w10 = wl * wb; f.w11 = wr * wb;
  f.off = (yc * W + xc) * C;
  return f;
}

// packed fp32x2 arithmetic (sm_100 FFMA2/FADD2/FMUL2): halves the issue slots of the per-channel math
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 splat(float a) { return make_float2(a, a); }

struct Tap8 {
  float2 v[4];
};
// one 256-bit read-only load (sm_100 LDG.E.256): the 8 channels of a tap in a single request, so the
// C/8 lanes of a pixel fetch its C*4-byte tap segment with one L1 wavefront per 128-byte line
__device__ __forceinline__ Tap8 load_tap8(const float* p) {
  Tap8 t;
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(t.v[0].x), "=f"(t.v[0].y), "=f"(t.v[1].x), "=f"(t.v[1].y), "=f"(t.v[2].x), "=f"(t.v[2].y),
                 "=f"(t.v[3].x), "=f"(t.v[3].y)
               : "l"(p));
  return t;
}

// Mapping: a thread owns (pixel, 8 consecutive channels = one G8 group); the C/8 lanes of a pixel are adjacent
// in the warp (C = 8: one thread per pixel, no cross-lane traffic at all).  Depth hypotheses are processed in
// chunks of DCH; inside a chunk the loop order is (source view, depth):
//   * the lanes of a pixel split the DCH projections of (view, chunk) between them and publish the footprints
//     through shared memory, so the ~60-instruction projection is computed once per (pixel, view, depth);
//   * walking depth innermost, consecutive hypotheses of the cascade's later stages land in the same 2x2 tap
//     block most of the time (sub-pixel steps along the epipolar line): the taps stay in registers and are
//     only re-fetched when the block changes;
//   * the per-channel math runs on packed fp32x2 instructions.
template <int C, int MODE, typename OutT, int DCH>
__global__ void __launch_bounds__(128) warp_agg_kernel(const WarpAggParams P) {
  constexpr int LPP = C / 8;     // lanes per pixel
  constexpr int PPW = 32 / LPP;  // pixels per warp (along x)
  constexpr int TW = PPW, TH = 4;  // 4 warps, one pixel row each
  constexpr int NPJ = (DCH + LPP - 1) / LPP;
  __shared__ float s_rt[kMaxSrc * 12];
  __shared__ float s_wnet[C + 5];
  __shared__ float4 s_fw[LPP > 1 ? 4 : 1][LPP > 1 ? PPW : 1][DCH + 1];
  __shared__ int s_fo[LPP > 1 ? 4 : 1][LPP > 1 ? PPW : 1][DCH + 1];

  const int b = blockIdx.z;
  const int H = P.H, W = P.W, D = P.D, n_src = P.n_src;
  for (int i = threadIdx.x; i < n_src * 12; i += blockDim.x) {
    int v = i / 12, j = i - v * 12;
    s_rt[i] = P.rot_trans[((long long)v * P.B + b) * 12 + j];
  }
  if (MODE == DAMVS_AGG_ADAPTIVE)
    for (int i = threadIdx.x; i < C + 5; i += blockDim.x) s_wnet[i] = P.wnet[i];
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane % LPP;  // channel group
  const int pw = lane / LPP; // pixel within the warp
  const int px = blockIdx.x * TW + pw;
  const int py = blockIdx.y * TH + warp;
  const bool live = px < W && py < H;
  const int x = live ? px : 0, y = live ? py : 0;
  const int c0 = q * 8;
  const long long HW = (long long)H * W;
  const long long img_stride = HW * C;

  const Tap8 rf = load_tap8(P.ref + (long long)b * img_stride + ((long long)y * W + x) * C + c0);
  const float fx = (float)x, fy = (float)y;
  const float inv_half_w = 1.f / (float)((W - 1) / 2.0), inv_half_h = 1.f / (float)((H - 1) / 2.0);
  const float fw = (float)W, fh = (float)H;
  float2 w1[4];
  float s1 = 0.f, b1 = 0.f, w2 = 0.f, s2 = 0.f, b2 = 0.f;
  if (MODE == DAMVS_AGG_ADAPTIVE) {
#pragma unroll
    for (int j = 0; j < 4; ++j) w1[j] = make_float2(s_wnet[c0 + 2 * j], s_wnet[c0 + 2 * j + 1]);
    s1 = s_wnet[C]; b1 = s_wnet[C + 1]; w2 = s_wnet[C + 2]; s2 = s_wnet[C + 3]; b2 = s_wnet[C + 4];
  }
  const float* hyp = P.per_pixel ? P.hyp + (long long)b * D * HW + (long long)y * W + x : P.hyp + (long long)b * D;
  const long long hyp_stride = P.per_pixel ? HW : 1;
  OutT* out = reinterpret_cast<OutT*>(P.out) + g8_offset(b, q, 0, y, x, C / 8, D, H, W);
  const long long out_stride = HW * 8;
  const float inv_n = 1.f / (float)(n_src + 1), inv_nsrc = 1.f / (float)n_src;

  for (int d0 = 0; d0 < D; d0 += DCH) {
    float2 acc[DCH][4], sq[MODE == DAMVS_AGG_VARIANCE ? DCH : 1][4];
#pragma unroll
    for (int j = 0; j < DCH; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (MODE == DAMVS_AGG_VARIANCE) {
          acc[j][k] = rf.v[k];
          sq[j][k] = mul2(rf.v[k], rf.v[k]);
        } else {
          acc[j][k] = make_float2(0.f, 0.f);
        }
      }
    // hypotheses this lane projects: j = q, q + LPP, ...
    float dep[NPJ];
#pragma unroll
    for (int k = 0; k < NPJ; ++k) {
      const int j = q + k * LPP, d = d0 + j;
      dep[k] = (j < DCH && d < D) ? __ldg(hyp + d * hyp_stride) : 1.f;
    }
    for (int v = 0; v < n_src; ++v) {
      const float* rt = s_rt + v * 12;
      // rot @ [x, y, 1]  (models/module.py:317)
      const float rx = fmaf(rt[0], fx, fmaf(rt[1], fy, rt[2]));
      const float ry = fmaf(rt[3], fx, fmaf(rt[4], fy, rt[5]));
      const float rz = fmaf(rt[6], fx, fmaf(rt[7], fy, rt[8]));
      Footprint fp[LPP > 1 ? 1 : DCH];
#pragma unroll
      for (int k = 0; k < NPJ; ++k) {
        const int j = q + k * LPP;
        if (j < DCH) {
          float ix, iy;
          project(rt, rx, ry, rz, dep[k], inv_half_w, inv_half_h, fw, fh, ix, iy);
          const Footprint f = make_footprint(ix, iy, H, W, C);
          if (LPP > 1) {
            s_fw[warp][pw][j] = make_float4(f.w00, f.w01, f.w10, f.w11);
            s_fo[warp][pw][j] = f.off;
          } else {
            fp[k] = f;
          }
        }
      }
      if (LPP > 1) __syncwarp();
      const float* img = P.src[v] + (long long)b * img_stride + c0;
      int cur = -1;
      Tap8 t00, t01, t10, t11;
#pragma unroll
      for (int k = 0; k < 4; ++k) t00.v[k] = t01.v[k] = t10.v[k] = t11.v[k] = make_float2(0.f, 0.f);
#pragma unroll
      for (int j = 0; j < DCH; ++j) {
        if (d0 + j < D) {  // uniform
          float4 fwt;
          int off;
          if (LPP > 1) {
            fwt = s_fw[warp][pw][j];
            off = s_fo[warp][pw][j];
          } else {
            fwt = make_float4(fp[j].w00, fp[j].w01, fp[j].w10, fp[j].w11);
            off = fp[j].off;
          }
          if (off != cur) {
            const float* p = img + off;
            t00 = load_tap8(p);
            t01 = load_tap8(p + C);
            t10 = load_tap8(p + (long long)W * C);
            t11 = load_tap8(p + (long long)W * C + C);
            cur = off;
          }
          const float2 a00 = splat(fwt.x), a01 = splat(fwt.y), a10 = splat(fwt.z), a11 = splat(fwt.w);
          float2 wv[4];
#pragma unroll
          for (int k = 0; k < 4; ++k)  // ATen grid_sampler_2d accumulation order: nw, ne, sw, se
            wv[k] = fma2(t11.v[k], a11, fma2(t10.v[k], a10, fma2(t01.v[k], a01, mul2(t00.v[k], a00))));
          if (MODE == DAMVS_AGG_VARIANCE) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              acc[j][k] = add2(acc[j][k], wv[k]);
              sq[j][k] = fma2(wv[k], wv[k], sq[j][k]);
            }
          } else {
            float2 e[4], sv = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 df = add2(rf.v[k], make_float2(-wv[k].x, -wv[k].y));
              e[k] = mul2(df, df);                 // cas_mvsnet.py:66
              sv = fma2(w1[k], e[k], sv);          // 1x1x1 conv C->1
            }
            float s = sv.x + sv.y;
#pragma unroll
            for (int o = LPP / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            const float a = fmaxf(s * s1 + b1, 0.f);                      // BN + ReLU
            const float2 wt = splat(fmaxf((a * w2) * s2 + b2, 0.f) + 1.f);  // conv 1->1, BN, ReLU; (weight + 1)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[j][k] = fma2(wt, e[k], acc[j][k]);   // cas_mvsnet.py:73-76
          }
        }
      }
      if (LPP > 1) __syncwarp();  // footprints of this view are consumed before the next view overwrites them
    }
#pragma unroll
    for (int j = 0; j < DCH; ++j) {
      if (d0 + j < D) {
        F8 r;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float2 a;
          if (MODE == DAMVS_AGG_VARIANCE) {
            const float2 m = mul2(acc[j][k], splat(inv_n));
            const float2 qn = mul2(sq[j][k], splat(inv_n));
            a = make_float2(qn.x - m.x * m.x, qn.y - m.y * m.y);   // cas_mvsnet.py:85
          } else {
            a = mul2(acc[j][k], splat(inv_nsrc));                  // cas_mvsnet.py:87
          }
          r.v[2 * k] = a.x; r.v[2 * k + 1] = a.y;
        }
        if (live) store8(out + (long long)(d0 + j) * out_stride, r);
      }
    }
  }
}

// stand-alone homo_warping: [B,H,W,C] -> [B,C,D,H,W] fp32 (reference output layout)
__global__ void __launch_bounds__(256) homo_warp_kernel(const float* __restrict__ src, const float* __restrict__ rot_trans,
                                                        const float* __restrict__ hyp, float* __restrict__ out,
                                                        int C, int D, int H, int W, int per_pixel) {
  const int b = blockIdx.z;
  const long long HW = (long long)H * W;
  long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= HW) return;
  const int d = blockIdx.y;
  const int y = (int)(pix / W), x = (int)(pix - (long long)y * W);
  float rt[12];
#pragma unroll
  for (int j = 0; j < 12; ++j) rt[j] = __ldg(rot_trans + b * 12 + j);
  const float fx = (float)x, fy = (float)y;
  float rx = fmaf(rt[0], fx, fmaf(rt[1], fy, rt[2]));
  float ry = fmaf(rt[3], fx, fmaf(rt[4], fy, rt[5]));
  float rz = fmaf(rt[6], fx, fmaf(rt[7], fy, rt[8]));
  float dep = per_pixel ? __ldg(hyp + ((long long)b * D + d) * HW + pix) : __ldg(hyp + b * D + d);
  float ix, iy;
  project(rt, rx, ry, rz, dep, 1.f / (float)((W - 1) / 2.0), 1.f / (float)((H - 1) / 2.0), (float)W, (float)H, ix, iy);
  const float* img = src + (long long)b * HW * C;
  float* o = out + (((long long)b * C) * D + d) * HW + pix;
  for (int c0 = 0; c0 < C; c0 += 4) {
    float4 v = sample4(img, H, W, C, c0, ix, iy);
    o[(long long)(c0 + 0) * D * HW] = v.x;
    o[(long long)(c0 + 1) * D * HW] = v.y;
    o[(long long)(c0 + 2) * D * HW] = v.z;
    o[(long long)(c0 + 3) * D * HW] = v.w;
  }
}

template <int C, int MODE>
static int launch_warp_agg(const WarpAggParams& P, int out_dtype, cudaStream_t st) {
  constexpr int TW = 32 / (C / 8), TH = 4, DCH = 4;
  dim3 grid((P.W + TW - 1) / TW, (P.H + TH - 1) / TH, P.B);
  if (out_dtype == DAMVS_F32)
    warp_agg_kernel<C, MODE, float, DCH><<<grid, 128, 0, st>>>(P);
  else if (out_dtype == DAMVS_F16)
    warp_agg_kernel<C, MODE, __half, DCH><<<grid, 128, 0, st>>>(P);
  else
    warp_agg_kernel<C, MODE, __nv_bfloat16, DCH><<<grid, 128, 0, st>>>(P);
  DAMVS_LAUNCH_OK("warp_agg kernel");
  return DAMVS_OK;
}

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_warp_agg_fwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src,
                                  const float* rot_trans, const float* depth_hyp, const float* wnet, void* out_vol,
                                  int B, int C, int D, int H, int W, int mode, int per_pixel_hyp, int out_dtype,
                                  void* stream) {
  DAMVS_REQUIRE(ref_nhwc && src_nhwc && rot_trans && depth_hyp && out_vol, "warp_agg: null pointer");
  DAMVS_REQUIRE(n_src >= 1 && n_src <= kMaxSrc, "warp_agg: n_src=%d outside [1,%d]", n_src, kMaxSrc);
  DAMVS_REQUIRE(B > 0 && D > 0 && H > 1 && W > 1, "warp_agg: bad shape B=%d D=%d H=%d W=%d (H, W >= 2)", B, D, H, W);
  DAMVS_REQUIRE(B <= 65535, "warp_agg: B too large");
  DAMVS_REQUIRE(mode == DAMVS_AGG_VARIANCE || mode == DAMVS_AGG_ADAPTIVE, "warp_agg: bad mode %d", mode);
  DAMVS_REQUIRE(mode == DAMVS_AGG_VARIANCE || wnet != nullptr, "warp_agg: adaptive mode needs wnet");
  DAMVS_REQUIRE(out_dtype == DAMVS_F32 || out_dtype == DAMVS_BF16 || out_dtype == DAMVS_F16, "warp_agg: bad out_dtype %d", out_dtype);
  DAMVS_REQUIRE((reinterpret_cast<uintptr_t>(ref_nhwc) & 31u) == 0 && aligned16(out_vol), "warp_agg: ref must be 32-byte, out 16-byte aligned");
  WarpAggParams P;
  P.ref = ref_nhwc;
  for (int v = 0; v < kMaxSrc; ++v) P.src[v] = v < n_src ? src_nhwc[v] : nullptr;
  for (int v = 0; v < n_src; ++v)
    DAMVS_REQUIRE(src_nhwc[v] && (reinterpret_cast<uintptr_t>(src_nhwc[v]) & 31u) == 0, "warp_agg: src[%d] null or not 32-byte aligned", v);
  P.rot_trans = rot_trans; P.hyp = depth_hyp; P.wnet = wnet; P.out = out_vol;
  P.B = B; P.n_src = n_src; P.D = D; P.H = H; P.W = W; P.per_pixel = per_pixel_hyp;
  cudaStream_t st = (cudaStream_t)stream;
#define DISPATCH(CC)                                                                          \
  case CC:                                                                                    \
    return mode == DAMVS_AGG_ADAPTIVE ? launch_warp_agg<CC, DAMVS_AGG_ADAPTIVE>(P, out_dtype, st) \
                                      : launch_warp_agg<CC, DAMVS_AGG_VARIANCE>(P, out_dtype, st);
  switch (C) {
    DISPATCH(8)
    DISPATCH(16)
    DISPATCH(32)
    DISPATCH(64)
    default:
      return set_error(DAMVS_ERR_UNSUPPORTED, "warp_agg: C=%d not in {8,16,32,64}", C);
  }
#undef DISPATCH
}

extern "C" int damvs_homo_warp_fwd(const float* src_nhwc, const float* rot_trans, const float* depth_hyp,
                                   float* out, int B, int C, int D, int H, int W, int per_pixel_hyp, void* stream) {
  DAMVS_REQUIRE(src_nhwc && rot_trans && depth_hyp && out, "homo_warp: null pointer");
  DAMVS_REQUIRE(B > 0 && C > 0 && C % 4 == 0 && D > 0 && H > 0 && W > 0, "homo_warp: bad shape (C must be a multiple of 4)");
  DAMVS_REQUIRE(D <= 65535 && B <= 65535, "homo_warp: D or B too large");
  DAMVS_REQUIRE(aligned16(src_nhwc), "homo_warp: src must be 16-byte aligned");
  long long HW = (long long)H * W;
  dim3 grid((unsigned)((HW + 255) / 256), D, B);
  homo_warp_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src_nhwc, rot_trans, depth_hyp, out, C, D, H, W,
                                                           per_pixel_hyp);
  DAMVS_LAUNCH_OK("homo_warp kernel");
  return DAMVS_OK;
}
