// Fused homography warp + multi-view aggregation, half-precision feature path (the bf16 pipeline's producer).
//
// Same operation as warp_agg.cu (reference models/cas_mvsnet.py:30-87, models/module.py:297-332, 544-563) for the
// `bf16` precision mode, where the cost volume is emitted in bf16 and the exact-rounding replication of the
// reference's coordinate arithmetic buys nothing.  What changes against the fp32 kernel, each measured there as a
// limiter (profiles/r01_ncu_summary_mid_round.md: 110-163 instructions per (view, voxel, 8 channels), L1 at 75 %):
//   * features are fp16 NHWC (damvs_nchw_to_nhwc_f16): a bilinear tap of 8 channels is ONE 16-byte load, half the
//     L1/L2 gather traffic of fp32;
//   * the blend runs on FHFMA (PTX fma.rn.f32.f16: fp16 operands selected straight out of the packed registers,
//     fp32 accumulate), so there is no unpack and the accumulation keeps fp32 precision; the first FMA of the chain
//     starts from -ref, which makes the chain's result the difference (ref - warp) up to sign;
//   * the projection is 3 FMA + 1 MUFU.RCP + 2 FMA per (pixel, view, hypothesis): the (W-1)/2 normalisation and the
//     align_corners=False un-normalisation of the reference collapse to ix = u * W/(W-1) - 0.5, with the scale folded
//     into the projection rows once per CTA;
//   * footprints (packed fp16 weights + byte offset, 16 bytes) are exchanged between the lanes of a pixel through
//     shared memory in a [depth][pixel] layout, one conflict-free LDS.128 per use.
// Kept from the fp32 kernel: thread = (pixel, 8 channels), depth chunks with (view, depth) loop order, packed fp32x2
// math after the blend, 16-byte stores.  Unlike the fp32 kernel, every hypothesis loads its taps (see HCfg).
//
// Sampling semantics are unchanged (zero padding per tap, no z > 0 mask, NaN coordinates sample zero); coordinates
// differ from the reference's by fp32 rounding only (<= 1e-4 pixel at W = 1600).
#include <cuda_fp16.h>

#include "common.cuh"

namespace damvs {

constexpr int kMaxSrcH = 15;
constexpr int kAggGwc = 2;   // internal MODE value: group-wise correlation (not in the reference; damvs_warp_gwc_fwd)

struct WarpAggHParams {
  const __half* ref;
  const __half* src[kMaxSrcH];
  const float* rot_trans;  // [n_src][B][12]
  const float* hyp;        // [B][D][H][W] or [B][D]
  const float* wnet;       // [C+5] or null
  void* out;               // G8 [B][C/8][D][H][W][8]
  int B, n_src, D, H, W, per_pixel;
};

// one bilinear footprint: fp16 weights (w00,w01 | w10,w11) and the byte offset of the (clamped) 2x2 block
struct FootH {
  uint32_t w01, w23;
  int off;
};

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

template <int C>
__device__ __forceinline__ FootH make_foot(float ix, float iy, int H, int W) {
  FootH f;
  const float fx0 = floorf(ix), fy0 = floorf(iy);
  float wr = ix - fx0, wb = iy - fy0;
  float wl = 1.f - wr, wt = 1.f - wb;
  int x0 = (int)fx0, y0 = (int)fy0;
  if ((unsigned)x0 >= (unsigned)(W - 1) || (unsigned)y0 >= (unsigned)(H - 1)) {
    // border / outside / NaN: clamp the block into the image and zero the weights of out-of-range taps
    if (!(ix > -1.f && ix < (float)W && iy > -1.f && iy < (float)H)) {
      wl = wr = wt = wb = 0.f;
      x0 = y0 = 0;
    } else {
      if (x0 < 0) { x0 = 0; wl = wr; wr = 0.f; } else if (x0 > W - 2) { x0 = W - 2; wr = wl; wl = 0.f; }
      if (y0 < 0) { y0 = 0; wt = wb; wb = 0.f; } else if (y0 > H - 2) { y0 = H - 2; wb = wt; wt = 0.f; }
    }
  }
  f.w01 = pack_h2(wl * wt, wr * wt);
  f.w23 = pack_h2(wl * wb, wr * wb);
  f.off = (y0 * W + x0) * (C * 2);
  return f;
}

// out = tap * w + in for 8 fp16 channels packed in a uint4 (FHFMA: fp16 operands, fp32 accumulate); w is the low
// (HI = false) or high half of `wpair`.  out and in may be the same array.
template <bool HI>
__device__ __forceinline__ void fhfma8(float (&out)[8], const float (&in)[8], const uint4& t, uint32_t wpair) {
  const uint32_t tw[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (HI) {
      asm("{.reg .b16 tl, th, wl, wh;\n\t"
          "mov.b32 {tl, th}, %4;\n\t"
          "mov.b32 {wl, wh}, %5;\n\t"
          "fma.rn.f32.f16 %0, tl, wh, %2;\n\t"
          "fma.rn.f32.f16 %1, th, wh, %3;}"
          : "=f"(out[2 * k]), "=f"(out[2 * k + 1]) : "f"(in[2 * k]), "f"(in[2 * k + 1]), "r"(tw[k]), "r"(wpair));
    } else {
      asm("{.reg .b16 tl, th, wl, wh;\n\t"
          "mov.b32 {tl, th}, %4;\n\t"
          "mov.b32 {wl, wh}, %5;\n\t"
          "fma.rn.f32.f16 %0, tl, wl, %2;\n\t"
          "fma.rn.f32.f16 %1, th, wl, %3;}"
          : "=f"(out[2 * k]), "=f"(out[2 * k + 1]) : "f"(in[2 * k]), "f"(in[2 * k + 1]), "r"(tw[k]), "r"(wpair));
    }
  }
}

__device__ __forceinline__ void store1(float* p, float v) { *p = v; }
__device__ __forceinline__ void store1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void store1(__half* p, float v) { *reinterpret_cast<unsigned short*>(p) = (unsigned short)(pack_f16x2(v, 0.f) & 0xffffu); }

__device__ __forceinline__ uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

template <int C, int MODE, typename OutT, int DCH, int MINB, bool FULL, int G = 0>
__global__ void __launch_bounds__(128, MINB) warp_agg_h_kernel(const WarpAggHParams P) {
  // group-wise correlation (MODE == kAggGwc): G groups of GS channels; a thread's 8 channels cover NV groups,
  // or an eighth / quarter / half of one group that LPG adjacent lanes finish with shuffles
  constexpr int GS = G > 0 ? C / G : 8;
  constexpr int NV = GS >= 8 ? 1 : 8 / GS;
  constexpr int LPG = GS >= 8 ? GS / 8 : 1;
  constexpr int GOUT = G > 0 && G < 8 ? 8 : (G > 0 ? G : 8);
  static_assert(MODE != kAggGwc || G > 0, "group-wise correlation needs a group count");
  constexpr int LPP = C / 8;       // lanes per pixel
  constexpr int PPW = 32 / LPP;    // pixels per warp (along x)
  constexpr int TW = PPW, TH = 4;
  constexpr int NPJ = (DCH + LPP - 1) / LPP;
  __shared__ float s_rt[kMaxSrcH * 12];
  __shared__ float s_wnet[C + 5];
  __shared__ uint4 s_fp[LPP > 1 ? 4 : 1][LPP > 1 ? DCH : 1][LPP > 1 ? PPW : 1];

  const int b = blockIdx.z;
  const int H = P.H, W = P.W, D = P.D, n_src = P.n_src;
  {
    // ix = u * W/(W-1) - 0.5: fold the scales into rows 0/1 of [rot | trans]
    const float sx = (float)W / (float)(W - 1), sy = (float)H / (float)(H - 1);
    for (int i = threadIdx.x; i < n_src * 12; i += blockDim.x) {
      const int v = i / 12, j = i - v * 12;
      const float s = (j < 3 || j == 9) ? sx : ((j < 6 || j == 10) ? sy : 1.f);
      s_rt[i] = P.rot_trans[((long long)v * P.B + b) * 12 + j] * s;
    }
  }
  if (MODE == DAMVS_AGG_ADAPTIVE)
    for (int i = threadIdx.x; i < C + 5; i += blockDim.x) s_wnet[i] = P.wnet[i];
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane % LPP, pw = lane / LPP;
  const int px = blockIdx.x * TW + pw, py = blockIdx.y * TH + warp;
  const bool live = px < W && py < H;
  const int x = live ? px : 0, y = live ? py : 0;
  const long long HW = (long long)H * W;
  const size_t img_bytes = (size_t)HW * C * 2;

  // -ref in fp32: the blend chain starts from it, so the chain ends in (warp - ref)
  float nrf[8];
  {
    const uint4 r = ldg16(reinterpret_cast<const char*>(P.ref) + (size_t)b * img_bytes + ((size_t)y * W + x) * (C * 2) + q * 16);
    const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f = __half22float2(h[k]);
      nrf[2 * k] = -f.x; nrf[2 * k + 1] = -f.y;
    }
  }
  const float fx = (float)x, fy = (float)y;
  float2 w1[4];
  float s1 = 0.f, b1 = 0.f, w2 = 0.f, s2 = 0.f, b2 = 0.f;
  if (MODE == DAMVS_AGG_ADAPTIVE) {
#pragma unroll
    for (int j = 0; j < 4; ++j) w1[j] = make_float2(s_wnet[q * 8 + 2 * j], s_wnet[q * 8 + 2 * j + 1]);
    s1 = s_wnet[C]; b1 = s_wnet[C + 1]; w2 = s_wnet[C + 2]; s2 = s_wnet[C + 3]; b2 = s_wnet[C + 4];
  }
  const float* hyp = P.per_pixel ? P.hyp + (long long)b * D * HW + (long long)y * W + x : P.hyp + (long long)b * D;
  const long long hyp_stride = P.per_pixel ? HW : 1;
  OutT* out = reinterpret_cast<OutT*>(P.out) + g8_offset(b, q, 0, y, x, C / 8, D, H, W);
  const long long out_stride = HW * 8;
  const float inv_n = 1.f / (float)(n_src + 1), inv_nsrc = 1.f / (float)n_src;

  for (int d0 = 0; d0 < D; d0 += DCH) {
    float2 acc[DCH][4], sq[MODE == DAMVS_AGG_VARIANCE ? DCH : 1][4];
    float accg[MODE == kAggGwc ? DCH : 1][NV];
    if (MODE == kAggGwc) {
#pragma unroll
      for (int j = 0; j < DCH; ++j)
#pragma unroll
        for (int k = 0; k < NV; ++k) accg[j][k] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < DCH; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (MODE == DAMVS_AGG_VARIANCE) {
          acc[j][k] = make_float2(-nrf[2 * k], -nrf[2 * k + 1]);
          sq[j][k] = make_float2(nrf[2 * k] * nrf[2 * k], nrf[2 * k + 1] * nrf[2 * k + 1]);
        } else {
          acc[j][k] = make_float2(0.f, 0.f);
        }
      }
    float dep[NPJ];
#pragma unroll
    for (int k = 0; k < NPJ; ++k) {
      const int j = q + k * LPP, d = d0 + j;
      dep[k] = (j < DCH && (FULL || d < D)) ? __ldg(hyp + d * hyp_stride) : 1.f;
    }
    for (int v = 0; v < n_src; ++v) {
      const float* rt = s_rt + v * 12;
      const float rx = fmaf(rt[0], fx, fmaf(rt[1], fy, rt[2]));
      const float ry = fmaf(rt[3], fx, fmaf(rt[4], fy, rt[5]));
      const float rz = fmaf(rt[6], fx, fmaf(rt[7], fy, rt[8]));
      FootH fp[LPP > 1 ? 1 : DCH];
#pragma unroll
      for (int k = 0; k < NPJ; ++k) {
        const int j = q + k * LPP;
        if (j < DCH) {
          const float pxs = fmaf(rx, dep[k], rt[9]), pys = fmaf(ry, dep[k], rt[10]), pz = fmaf(rz, dep[k], rt[11]);
          float inv;                          // MUFU.RCP (1 ulp); z = 0 gives inf/NaN -> samples zero
          asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(pz));
          const FootH f = make_foot<C>(fmaf(pxs, inv, -0.5f), fmaf(pys, inv, -0.5f), H, W);
          if (LPP > 1) s_fp[warp][j][pw] = make_uint4(f.w01, f.w23, (uint32_t)f.off, 0u);
          else fp[k] = f;
        }
      }
      if (LPP > 1) __syncwarp();
      const char* img = reinterpret_cast<const char*>(P.src[v]) + (size_t)b * img_bytes + q * 16;
#pragma unroll
      for (int j = 0; j < DCH; ++j) {
        if (FULL || d0 + j < D) {  // uniform
          FootH f;
          if (LPP > 1) {
            const uint4 u = s_fp[warp][j][pw];
            f.w01 = u.x; f.w23 = u.y; f.off = (int)u.z;
          } else {
            f = fp[j];
          }
          const char* p = img + f.off;
          const uint4 t00 = ldg16(p), t01 = ldg16(p + C * 2);
          const uint4 t10 = ldg16(p + (size_t)W * (C * 2)), t11 = ldg16(p + (size_t)W * (C * 2) + C * 2);
          float df[8], base[8];   // warp - ref  (variance mode: warp)
#pragma unroll
          for (int k = 0; k < 8; ++k) base[k] = MODE == DAMVS_AGG_ADAPTIVE ? nrf[k] : 0.f;
          fhfma8<false>(df, base, t00, f.w01);
          fhfma8<true>(df, df, t01, f.w01);
          fhfma8<false>(df, df, t10, f.w23);
          fhfma8<true>(df, df, t11, f.w23);
          if (MODE == kAggGwc) {
            float pr[8];                                   // ref * warp (nrf holds -ref)
#pragma unroll
            for (int k = 0; k < 8; ++k) pr[k] = -nrf[k] * df[k];
            if (GS >= 8) {
              float s = ((pr[0] + pr[1]) + (pr[2] + pr[3])) + ((pr[4] + pr[5]) + (pr[6] + pr[7]));
#pragma unroll
              for (int o = LPG / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
              accg[j][0] += s;
            } else {
#pragma unroll
              for (int k = 0; k < NV; ++k) {
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < GS; ++i) s += pr[k * GS + i];
                accg[j][k] += s;
              }
            }
          } else if (MODE == DAMVS_AGG_VARIANCE) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 d2 = make_float2(df[2 * k], df[2 * k + 1]);
              acc[j][k] = __fadd2_rn(acc[j][k], d2);
              sq[j][k] = __ffma2_rn(d2, d2, sq[j][k]);
            }
          } else {
            float2 e[4], sv = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 d2 = make_float2(df[2 * k], df[2 * k + 1]);
              e[k] = __fmul2_rn(d2, d2);                          // cas_mvsnet.py:66
              sv = __ffma2_rn(w1[k], e[k], sv);                   // 1x1x1 conv C->1
            }
            float s = sv.x + sv.y;
#pragma unroll
            for (int o = LPP / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            const float a = fmaxf(fmaf(s, s1, b1), 0.f);                       // BN + ReLU
            const float wtv = fmaxf(fmaf(a * w2, s2, b2), 0.f) + 1.f;         // conv 1->1, BN, ReLU; (weight + 1)
            const float2 wt = make_float2(wtv, wtv);
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[j][k] = __ffma2_rn(wt, e[k], acc[j][k]);   // cas_mvsnet.py:73-76
          }
        }
      }
      if (LPP > 1) __syncwarp();  // footprints of this view are consumed before the next view overwrites them
    }
    if (MODE == kAggGwc) {
      const float norm = 1.f / ((float)n_src * (float)GS);
      OutT* og = reinterpret_cast<OutT*>(P.out);
#pragma unroll
      for (int j = 0; j < DCH; ++j) {
        if (!(FULL || d0 + j < D) || !live) continue;
        if (GS >= 8) {
          if (q % LPG == 0) {
            const int ch = q / LPG;
            OutT* o = og + g8_offset(b, ch / 8, d0 + j, y, x, GOUT / 8, D, H, W) + (ch % 8);
            store1(o, accg[j][0] * norm);
            if (G < 8) store1(o + G, 0.f);                    // zero padding channels (G = 4)
          }
        } else {
          const int ch0 = q * NV;
          OutT* o = og + g8_offset(b, ch0 / 8, d0 + j, y, x, GOUT / 8, D, H, W) + (ch0 % 8);
          if (NV == 8) {
            F8 r;
#pragma unroll
            for (int k = 0; k < 8; ++k) r.v[k] = accg[j][k] * norm;
            store8(o, r);
          } else if (NV == 4) {
            store4(o, accg[j][0] * norm, accg[j][1] * norm, accg[j][2] * norm, accg[j][3] * norm);
          } else {
#pragma unroll
            for (int k = 0; k < NV; ++k) store1(o + k, accg[j][k] * norm);
          }
          if (G < 8) {
#pragma unroll
            for (int k = 0; k < NV; ++k) store1(o + G + k, 0.f);
          }
        }
      }
      continue;
    }
#pragma unroll
    for (int j = 0; j < DCH; ++j) {
      if (FULL || d0 + j < D) {
        F8 r;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float2 a;
          const float2 ac = acc[j][k];
          if (MODE == DAMVS_AGG_VARIANCE) {
            const float2 m = make_float2(ac.x * inv_n, ac.y * inv_n);
            const float2 qq = sq[j][k];
            a = make_float2(fmaf(qq.x, inv_n, -m.x * m.x), fmaf(qq.y, inv_n, -m.y * m.y));   // cas_mvsnet.py:85
          } else {
            a = make_float2(ac.x * inv_nsrc, ac.y * inv_nsrc);                                // cas_mvsnet.py:87
          }
          r.v[2 * k] = a.x; r.v[2 * k + 1] = a.y;
        }
        if (live) store8(out + (long long)(d0 + j) * out_stride, r);
      }
    }
  }
}

// in [B][C][HW] fp32 -> out [B][HW][C] fp16 (saturating).  Tiled transpose through shared memory: 16-byte loads along
// the pixel axis into an fp32 [C][128 + 1] tile, then thread (pixel, 8-channel group) -- groups fastest, so a warp's
// 16-byte stores are contiguous -- reads its 8 channels (pitch 129 makes the 32 lanes hit 32 different banks).
constexpr int kTP = 128;
constexpr int kTPitch = kTP + 1;
constexpr int kMaxRepack = 16;
struct RepackPtrs {
  const float* in[kMaxRepack];
  __half* out[kMaxRepack];
};
__global__ void __launch_bounds__(128) nchw_to_nhwc_f16_kernel(const __grid_constant__ RepackPtrs ptrs, int C, long long HW,
                                                               int tiles_per_cta) {
  extern __shared__ float ftile[];  // [C][kTPitch]
  const float* __restrict__ in = ptrs.in[blockIdx.z];
  __half* __restrict__ out = ptrs.out[blockIdx.z];
  const int b = blockIdx.y, t = threadIdx.x;
  const bool vec = (HW % 4 == 0);
  const int cpp = C / 8;
  for (int it = 0; it < tiles_per_cta; ++it) {
    const long long p0 = ((long long)blockIdx.x * tiles_per_cta + it) * kTP;
    if (p0 >= HW) break;
    const int np = (int)min((long long)kTP, HW - p0);
    const float* src = in + (long long)b * C * HW + p0;
    if (vec) {
      for (int i = t; i < C * (kTP / 4); i += blockDim.x) {
        const int c = i / (kTP / 4), p4 = (i - c * (kTP / 4)) * 4;
        if (p4 < np) {
          const float4 v = __ldcs(reinterpret_cast<const float4*>(src + (long long)c * HW + p4));
          float* d = ftile + c * kTPitch + p4;
          d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        }
      }
    } else {
      for (int i = t; i < C * kTP; i += blockDim.x) {
        const int c = i / kTP, p = i - c * kTP;
        if (p < np) ftile[c * kTPitch + p] = __ldcs(src + (long long)c * HW + p);
      }
    }
    __syncthreads();
    for (int i = t; i < np * cpp; i += blockDim.x) {
      const int p = i / cpp, g = i - p * cpp;
      const float* s0 = ftile + (g * 8) * kTPitch + p;
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float lo = fminf(fmaxf(s0[(2 * k) * kTPitch], -65504.f), 65504.f);
        const float hi = fminf(fmaxf(s0[(2 * k + 1) * kTPitch], -65504.f), 65504.f);
        w[k] = pack_h2(lo, hi);
      }
      *reinterpret_cast<uint4*>(out + ((long long)b * HW + p0 + p) * C + g * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    __syncthreads();
  }
}

// Per channel width: depth chunk and minimum CTAs per SM (measured at the DTU-test stage shapes on B200: unconditional
// tap loads let the compiler batch a chunk's gathers, which beats skipping repeated 2x2 blocks; the narrow kernels trade
// accumulators for occupancy).  Eight channels per thread: 16 (two G8 groups per thread) saves ~30 % of the instructions
// but costs more in occupancy at 128 registers -- 488 vs 403 us at stage 1, 528 vs 515 us at stage 2.
template <int C> struct HCfg { static constexpr int DCH = 4, MINB = 1; };
template <> struct HCfg<32> { static constexpr int DCH = 4, MINB = 5; };
template <> struct HCfg<16> { static constexpr int DCH = 2, MINB = 6; };
template <> struct HCfg<8> { static constexpr int DCH = 2, MINB = 8; };

template <int C, int MODE>
static int launch_h(const WarpAggHParams& P, int out_dtype, cudaStream_t st) {
  constexpr int DCH = HCfg<C>::DCH, MINB = HCfg<C>::MINB;
  constexpr int TW = 32 / (C / 8), TH = 4;
  dim3 grid((P.W + TW - 1) / TW, (P.H + TH - 1) / TH, P.B);
  const bool full = P.D % DCH == 0;
  if (out_dtype == DAMVS_F32) warp_agg_h_kernel<C, MODE, float, DCH, 1, false><<<grid, 128, 0, st>>>(P);
  else if (out_dtype == DAMVS_F16 && full) warp_agg_h_kernel<C, MODE, __half, DCH, MINB, true><<<grid, 128, 0, st>>>(P);
  else if (out_dtype == DAMVS_F16) warp_agg_h_kernel<C, MODE, __half, DCH, MINB, false><<<grid, 128, 0, st>>>(P);
  else if (full) warp_agg_h_kernel<C, MODE, __nv_bfloat16, DCH, MINB, true><<<grid, 128, 0, st>>>(P);
  else warp_agg_h_kernel<C, MODE, __nv_bfloat16, DCH, MINB, false><<<grid, 128, 0, st>>>(P);
  DAMVS_LAUNCH_OK("warp_agg_h kernel");
  return DAMVS_OK;
}

// Group-wise correlation on the tuned kernel (fp16 features, 2-byte volume, D a multiple of the depth chunk); called by
// damvs_warp_gwc_fwd (warp_gwc.cu), which keeps the plain kernel for every other case.
template <int C, int G>
static int launch_gwc_fast_cg(const WarpAggHParams& P, int out_dtype, cudaStream_t st) {
  constexpr int DCH = HCfg<C>::DCH, MINB = HCfg<C>::MINB;
  constexpr int TW = 32 / (C / 8), TH = 4;
  dim3 grid((P.W + TW - 1) / TW, (P.H + TH - 1) / TH, P.B);
  if (out_dtype == DAMVS_F16) warp_agg_h_kernel<C, kAggGwc, __half, DCH, MINB, true, G><<<grid, 128, 0, st>>>(P);
  else warp_agg_h_kernel<C, kAggGwc, __nv_bfloat16, DCH, MINB, true, G><<<grid, 128, 0, st>>>(P);
  DAMVS_LAUNCH_OK("warp_agg_h kernel (group-wise correlation)");
  return DAMVS_OK;
}

bool warp_gwc_fast_supported(int C, int G, int D, int n_src, int feat_dtype, int out_dtype) {
  const int dch = C == 32 ? HCfg<32>::DCH : (C == 16 ? HCfg<16>::DCH : HCfg<8>::DCH);
  return feat_dtype == DAMVS_F16 && (out_dtype == DAMVS_F16 || out_dtype == DAMVS_BF16) && D % dch == 0 && n_src <= kMaxSrcH;
}

int warp_gwc_fast_launch(const void* ref, const void* const* src, int n_src, const float* rot_trans, const float* hyp, void* out, int B, int C,
                         int G, int D, int H, int W, int per_pixel, int out_dtype, cudaStream_t st) {
  WarpAggHParams P;
  P.ref = (const __half*)ref;
  for (int v = 0; v < kMaxSrcH; ++v) P.src[v] = v < n_src ? (const __half*)src[v] : nullptr;
  P.rot_trans = rot_trans; P.hyp = hyp; P.wnet = nullptr; P.out = out;
  P.B = B; P.n_src = n_src; P.D = D; P.H = H; P.W = W; P.per_pixel = per_pixel;
#define GO(CC, GG) if (C == CC && G == GG) return launch_gwc_fast_cg<CC, GG>(P, out_dtype, st)
  GO(8, 4); GO(8, 8);
  GO(16, 4); GO(16, 8); GO(16, 16);
  GO(32, 4); GO(32, 8); GO(32, 16); GO(32, 32);
#undef GO
  return set_error(DAMVS_ERR_UNSUPPORTED, "warp_gwc (fast): C=%d, G=%d not supported", C, G);
}

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_nchw_to_nhwc_f16_multi(const float* const* ins, void* const* outs, int n, int B, int C, int H, int W, void* stream) {
  DAMVS_REQUIRE(ins && outs, "nchw_to_nhwc_f16: null pointer");
  DAMVS_REQUIRE(n >= 1 && n <= kMaxRepack, "nchw_to_nhwc_f16: n=%d outside [1,%d]", n, kMaxRepack);
  DAMVS_REQUIRE(B > 0 && B <= 65535 && C > 0 && C % 8 == 0 && C <= 256 && H > 0 && W > 0, "nchw_to_nhwc_f16: bad shape (C must be a multiple of 8)");
  RepackPtrs ptrs{};
  for (int i = 0; i < n; ++i) {
    DAMVS_REQUIRE(ins[i] && outs[i] && aligned16(ins[i]) && aligned16(outs[i]), "nchw_to_nhwc_f16: tensor %d null or not 16-byte aligned", i);
    ptrs.in[i] = ins[i];
    ptrs.out[i] = (__half*)outs[i];
  }
  const long long HW = (long long)H * W;
  const long long tiles = (HW + kTP - 1) / kTP;
  const int tiles_per_cta = tiles * n > 148 * 32 ? 2 : 1;
  dim3 grid((unsigned)((tiles + tiles_per_cta - 1) / tiles_per_cta), B, n);
  const size_t smem = (size_t)C * kTPitch * sizeof(float);
  if (smem > 48 * 1024) DAMVS_CUDA_OK(cudaFuncSetAttribute(nchw_to_nhwc_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nchw_to_nhwc_f16_kernel<<<grid, 128, smem, (cudaStream_t)stream>>>(ptrs, C, HW, tiles_per_cta);
  DAMVS_LAUNCH_OK("nchw_to_nhwc_f16 kernel");
  return DAMVS_OK;
}

extern "C" int damvs_nchw_to_nhwc_f16(const float* in, void* out, int B, int C, int H, int W, void* stream) {
  const float* ins[1] = {in};
  void* outs[1] = {out};
  return damvs_nchw_to_nhwc_f16_multi(ins, outs, 1, B, C, H, W, stream);
}

extern "C" int damvs_warp_agg_fwd_f16(const void* ref_nhwc, const void* const* src_nhwc, int n_src, const float* rot_trans,
                                      const float* depth_hyp, const float* wnet, void* out_vol, int B, int C, int D, int H,
                                      int W, int mode, int per_pixel_hyp, int out_dtype, void* stream) {
  DAMVS_REQUIRE(ref_nhwc && src_nhwc && rot_trans && depth_hyp && out_vol, "warp_agg_f16: null pointer");
  DAMVS_REQUIRE(n_src >= 1 && n_src <= kMaxSrcH, "warp_agg_f16: n_src=%d outside [1,%d]", n_src, kMaxSrcH);
  DAMVS_REQUIRE(B > 0 && B <= 65535 && D > 0 && H > 1 && W > 1, "warp_agg_f16: bad shape B=%d D=%d H=%d W=%d (H, W >= 2)", B, D, H, W);
  DAMVS_REQUIRE((long long)H * W * C * 2 < (1ll << 31), "warp_agg_f16: feature map too large for 32-bit tap offsets");
  DAMVS_REQUIRE(mode == DAMVS_AGG_VARIANCE || mode == DAMVS_AGG_ADAPTIVE, "warp_agg_f16: bad mode %d", mode);
  DAMVS_REQUIRE(mode == DAMVS_AGG_VARIANCE || wnet != nullptr, "warp_agg_f16: adaptive mode needs wnet");
  DAMVS_REQUIRE(out_dtype == DAMVS_F32 || out_dtype == DAMVS_BF16 || out_dtype == DAMVS_F16, "warp_agg_f16: bad out_dtype %d", out_dtype);
  DAMVS_REQUIRE(aligned16(ref_nhwc) && aligned16(out_vol), "warp_agg_f16: ref and out must be 16-byte aligned");
  WarpAggHParams P;
  P.ref = (const __half*)ref_nhwc;
  for (int v = 0; v < kMaxSrcH; ++v) P.src[v] = v < n_src ? (const __half*)src_nhwc[v] : nullptr;
  for (int v = 0; v < n_src; ++v)
    DAMVS_REQUIRE(src_nhwc[v] && aligned16(src_nhwc[v]), "warp_agg_f16: src[%d] null or not 16-byte aligned", v);
  P.rot_trans = rot_trans; P.hyp = depth_hyp; P.wnet = wnet; P.out = out_vol;
  P.B = B; P.n_src = n_src; P.D = D; P.H = H; P.W = W; P.per_pixel = per_pixel_hyp;
  cudaStream_t st = (cudaStream_t)stream;
#define DISPATCH(CC)                                                                    \
  case CC:                                                                              \
    return mode == DAMVS_AGG_ADAPTIVE ? launch_h<CC, DAMVS_AGG_ADAPTIVE>(P, out_dtype, st) \
                                      : launch_h<CC, DAMVS_AGG_VARIANCE>(P, out_dtype, st);
  switch (C) {
    DISPATCH(8)
    DISPATCH(16)
    DISPATCH(32)
    DISPATCH(64)
    default:
      return set_error(DAMVS_ERR_UNSUPPORTED, "warp_agg_f16: C=%d not in {8,16,32,64}", C);
  }
#undef DISPATCH
}
