// Training forward and backward of the fused warp + GROUP-WISE CORRELATION aggregation (not in the reference; the
// inference kernel and its definition are in warp_gwc.cu).  With S = C/G channels per group, gamma(c) = c / S and
// k = 1 / (n_src * S):
//
//     vol[b,g,d,y,x] = k * sum_v sum_{c: gamma(c) = g} ref[b,y,x,c] * warp_v[b,y,x,c,d]
//
//     g_ref[b,y,x,c] = k * sum_d gv[b,gamma(c),d,y,x] * sum_v warp_v[b,y,x,c,d]                 (overwritten)
//     g_src_v        = bilinear scatter-add of k * gv[b,gamma(c),d,y,x] * ref[b,y,x,c]        (accumulated)
//
// The forward and the backward sample at the same coordinates: both use project_b / footprint_b / blend8 /
// scatter8 (warp_common.cuh), which keep the reference's operation order, so the gradient belongs to the function the
// forward evaluated.  The inference kernel folds the normalisation into the projection instead and is not used here.
// The sampling grid and the hypotheses get no gradient (reference models/module.py:307 builds the grid under no_grad).
// G = 4 volumes carry 8 channels; the forward writes channels 4..7 as zero and the backward never reads them.
//
// Mapping as warp_agg_bwd.cu: thread = (pixel, 8 channels), the C/8 lanes of a pixel adjacent in the warp.  Per
// (depth, view) one projection, one 4-tap blend and, in the backward, one 4-tap vector-atomic scatter: the scattered
// value k * gv * ref does not depend on the view, so it is formed once per depth.
#include "warp_common.cuh"

namespace damvs {

struct WarpGwcTrainParams {
  const float* ref;
  const float* src[kMaxSrcB];
  float* g_src[kMaxSrcB];
  const float* rot_trans;
  const float* hyp;
  void* vol;       // forward: out; backward: g_vol in (both G8, max(G, 8) channels)
  float* g_ref;    // backward: out
  int B, n_src, D, H, W, per_pixel;
};

__device__ __forceinline__ float ld1(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld1(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ void st1(float* p, float v) { *p = v; }
__device__ __forceinline__ void st1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// forward epilogue at one depth: group sums of ref * sum_v warp_v, scaled by k, into the G8 volume; `o` points at this
// thread's first group.  Groups wider than 8 channels are finished with xor-shuffles (all lanes take part).
template <int C, int G, typename VT>
__device__ __forceinline__ void store_groups(VT* o, const F8& rf, const float (&wsum)[8], float k, bool live, int q) {
  constexpr int GS = C / G, NV = GS >= 8 ? 1 : 8 / GS, LPG = GS >= 8 ? GS / 8 : 1;
  float pr[8], acc[NV];
#pragma unroll
  for (int j = 0; j < 8; ++j) pr[j] = rf.v[j] * wsum[j];
  if (GS >= 8) {
    float s = ((pr[0] + pr[1]) + (pr[2] + pr[3])) + ((pr[4] + pr[5]) + (pr[6] + pr[7]));
#pragma unroll
    for (int m = LPG / 2; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    acc[0] = s;
  } else {
#pragma unroll
    for (int t = 0; t < NV; ++t) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < GS; ++j) s += pr[t * GS + j];
      acc[t] = s;
    }
  }
  if (!live || q % LPG != 0) return;
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    st1(o + t, acc[t] * k);
    if (G < 8) st1(o + G + t, 0.f);   // padding channels G..7 of the single chunk
  }
}

template <int C, int G, bool BWD, typename VT>
__global__ void __launch_bounds__(128) warp_gwc_train_kernel(const WarpGwcTrainParams P) {
  constexpr int LPP = C / 8, PPW = 32 / LPP, TW = PPW, TH = 4;
  constexpr int GS = C / G;                   // channels per group
  constexpr int NV = GS >= 8 ? 1 : 8 / GS;    // groups a thread's 8 channels touch
  constexpr int GOUT = G < 8 ? 8 : G;         // channels of the volume
  __shared__ float s_rt[kMaxSrcB * 12];
  const int b = blockIdx.z, H = P.H, W = P.W, D = P.D, n_src = P.n_src;
  for (int i = threadIdx.x; i < n_src * 12; i += blockDim.x) s_rt[i] = P.rot_trans[((long long)(i / 12) * P.B + b) * 12 + i % 12];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane % LPP, pw = lane / LPP;
  const int px = blockIdx.x * TW + pw, py = blockIdx.y * TH + warp;
  const bool live = px < W && py < H;
  const int x = live ? px : 0, y = live ? py : 0, c0 = q * 8;
  const long long HW = (long long)H * W, img_stride = HW * C, pix = (long long)y * W + x;
  const F8 rf = load8(P.ref + (long long)b * img_stride + pix * C + c0);
  const float fx = (float)x, fy = (float)y, fw = (float)W, fh = (float)H;
  const float inv_half_w = 1.f / (float)((W - 1) / 2.0), inv_half_h = 1.f / (float)((H - 1) / 2.0);
  const float* hyp = P.per_pixel ? P.hyp + (long long)b * D * HW + pix : P.hyp + (long long)b * D;
  const long long hyp_stride = P.per_pixel ? HW : 1;
  const long long vol_stride = HW * 8;
  const float k = 1.f / ((float)n_src * (float)GS);
  // first group of this thread's channels and its place in the G8 volume (NV consecutive groups, one 8-channel chunk)
  const int g0 = GS >= 8 ? c0 / GS : q * NV;
  VT* vol = reinterpret_cast<VT*>(P.vol) + g8_offset(b, g0 / 8, 0, y, x, GOUT / 8, D, H, W) + g0 % 8;

  float gref[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) gref[j] = 0.f;

  for (int d = 0; d < D; ++d) {
    const float dep = __ldg(hyp + d * hyp_stride);
    float gsel[8], gsrc[8];
    if (BWD) {
      float gv[NV];
#pragma unroll
      for (int t = 0; t < NV; ++t) gv[t] = ld1(vol + d * vol_stride + t);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        gsel[j] = gv[j / (8 / NV)];            // upstream gradient of channel c0 + j's group
        gsrc[j] = k * gsel[j] * rf.v[j];       // what every view scatters at this depth
      }
    }
    float wsum[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) wsum[j] = 0.f;
    for (int v = 0; v < n_src; ++v) {
      float ix, iy, w[4], wv[8];
      project_b(s_rt + v * 12, fx, fy, dep, inv_half_w, inv_half_h, fw, fh, ix, iy);
      const int off = footprint_b(ix, iy, H, W, C, w);
      blend8(P.src[v] + (long long)b * img_stride + off + c0, W, C, w, wv);
#pragma unroll
      for (int j = 0; j < 8; ++j) wsum[j] += wv[j];
      if (BWD && live) scatter8(P.g_src[v] + (long long)b * img_stride + off + c0, W, C, w, gsrc);
    }
    if (BWD) {
#pragma unroll
      for (int j = 0; j < 8; ++j) gref[j] = fmaf(gsel[j], wsum[j], gref[j]);
    } else {
      store_groups<C, G>(vol + d * vol_stride, rf, wsum, k, live, q);
    }
  }
  if (BWD && live) {
    F8 r;
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] = k * gref[j];
    store8(P.g_ref + (long long)b * img_stride + pix * C + c0, r);
  }
}

template <int C, int G, bool BWD>
static int launch_gwc_train(const WarpGwcTrainParams& P, int vdtype, cudaStream_t st) {
  constexpr int TW = 32 / (C / 8), TH = 4;
  dim3 grid((P.W + TW - 1) / TW, (P.H + TH - 1) / TH, P.B);
  if (vdtype == DAMVS_BF16) warp_gwc_train_kernel<C, G, BWD, __nv_bfloat16><<<grid, 128, 0, st>>>(P);
  else warp_gwc_train_kernel<C, G, BWD, float><<<grid, 128, 0, st>>>(P);
  DAMVS_LAUNCH_OK(BWD ? "warp_gwc_bwd kernel" : "warp_gwc_train_fwd kernel");
  return DAMVS_OK;
}

template <bool BWD>
static int dispatch_gwc_train(const WarpGwcTrainParams& P, int C, int G, int vdtype, cudaStream_t st) {
#define GO(CC, GG) if (C == CC && G == GG) return launch_gwc_train<CC, GG, BWD>(P, vdtype, st)
  GO(8, 4); GO(8, 8);
  GO(16, 4); GO(16, 8); GO(16, 16);
  GO(32, 4); GO(32, 8); GO(32, 16); GO(32, 32);
#undef GO
  return set_error(DAMVS_ERR_UNSUPPORTED, "warp_gwc_train: C=%d, G=%d not supported (C in {8,16,32}, G in {4,8,16,32}, G <= C)", C, G);
}

// host-side checks shared by both entry points; g_src == nullptr for the forward
static int fill_gwc_train(WarpGwcTrainParams& P, const char* name, const float* ref, const float* const* src, float* const* g_src,
                          int n_src, const float* rot_trans, const float* hyp, const void* vol, int vdtype, int B, int C, int G,
                          int D, int H, int W, int per_pixel) {
  DAMVS_REQUIRE(ref && src && rot_trans && hyp && vol, "%s: null pointer", name);
  DAMVS_REQUIRE(n_src >= 1 && n_src <= kMaxSrcB, "%s: n_src=%d outside [1,%d]", name, n_src, kMaxSrcB);
  DAMVS_REQUIRE(B > 0 && B <= 65535 && D > 0 && H > 1 && W > 1, "%s: bad shape B=%d D=%d H=%d W=%d (H, W >= 2)", name, B, D, H, W);
  if (!((C == 8 || C == 16 || C == 32) && (G == 4 || G == 8 || G == 16 || G == 32) && G <= C))
    return set_error(DAMVS_ERR_UNSUPPORTED, "%s: C=%d, G=%d not supported (C in {8,16,32}, G in {4,8,16,32}, G <= C)", name, C, G);
  DAMVS_REQUIRE((long long)H * W * C < (1ll << 31), "%s: feature map too large for 32-bit tap offsets", name);
  DAMVS_REQUIRE(vdtype == DAMVS_F32 || vdtype == DAMVS_BF16, "%s: volume dtype %d is neither fp32 nor bf16", name, vdtype);
  DAMVS_REQUIRE(aligned16(ref) && aligned16(vol), "%s: ref and the volume must be 16-byte aligned", name);
  P = WarpGwcTrainParams{};
  P.ref = ref;
  for (int v = 0; v < n_src; ++v) {
    DAMVS_REQUIRE(src[v] && aligned16(src[v]), "%s: src[%d] null or misaligned", name, v);
    P.src[v] = src[v];
    if (g_src) {
      DAMVS_REQUIRE(g_src[v] && aligned16(g_src[v]), "%s: g_src[%d] null or misaligned", name, v);
      P.g_src[v] = g_src[v];
    }
  }
  P.rot_trans = rot_trans; P.hyp = hyp; P.vol = const_cast<void*>(vol);
  P.B = B; P.n_src = n_src; P.D = D; P.H = H; P.W = W; P.per_pixel = per_pixel;
  return DAMVS_OK;
}

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_warp_gwc_train_fwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                                        const float* depth_hyp, void* out_vol, int B, int C, int G, int D, int H, int W,
                                        int per_pixel_hyp, int out_dtype, void* stream) {
  WarpGwcTrainParams P;
  int rc = fill_gwc_train(P, "warp_gwc_train_fwd", ref_nhwc, src_nhwc, nullptr, n_src, rot_trans, depth_hyp, out_vol, out_dtype, B, C,
                          G, D, H, W, per_pixel_hyp);
  if (rc) return rc;
  return dispatch_gwc_train<false>(P, C, G, out_dtype, (cudaStream_t)stream);
}

extern "C" int damvs_warp_gwc_bwd(const float* ref_nhwc, const float* const* src_nhwc, int n_src, const float* rot_trans,
                                  const float* depth_hyp, const void* g_vol, int g_dtype, float* g_ref, float* const* g_src, int B,
                                  int C, int G, int D, int H, int W, int per_pixel_hyp, void* stream) {
  DAMVS_REQUIRE(g_ref && g_src, "warp_gwc_bwd: null pointer");
  DAMVS_REQUIRE(aligned16(g_ref), "warp_gwc_bwd: g_ref must be 16-byte aligned");
  WarpGwcTrainParams P;
  int rc = fill_gwc_train(P, "warp_gwc_bwd", ref_nhwc, src_nhwc, g_src, n_src, rot_trans, depth_hyp, g_vol, g_dtype, B, C, G, D, H, W,
                          per_pixel_hyp);
  if (rc) return rc;
  P.g_ref = g_ref;
  return dispatch_gwc_train<true>(P, C, G, g_dtype, (cudaStream_t)stream);
}
