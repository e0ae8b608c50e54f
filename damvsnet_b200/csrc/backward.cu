// Backward kernels of the hot path: regression head and convolution weight gradients.
//
// The reference's backward is PyTorch autograd through softmax / regression, nn.Conv3d /
// nn.ConvTranspose3d / BatchNorm3d (reference models/module.py:117-202, 510-541) and the hypothesis
// variance (models/cas_mvsnet.py:105-124).  Here:
//   * head_bwd_kernel        closed-form gradient of depth / variance / prob_volume w.r.t. the logits
//                            (and optionally the hypotheses), SURVEY.md section 3.2;
//   * (BatchNorm + ReLU backward lives in bn.cu)
//   * conv_wgrad_kernel      dW[co][ci][tap] = sum_voxels g_y[co](o) * x[ci](i(o, tap)) (CUDA cores, fp32 atomics).
// The data gradient of a conv block is one more forward-type convolution (transposed roles), run by the
// existing conv kernels with re-packed weights -- see damvsnet_b200/autograd.py.
#include <algorithm>

#include "common.cuh"

namespace damvs {

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ prob, const float* __restrict__ hyp,
                                                       const float* __restrict__ depth, const float* __restrict__ g_depth,
                                                       const float* __restrict__ g_var, const float* __restrict__ g_prob,
                                                       float* __restrict__ g_logits, float* __restrict__ g_hyp, int D,
                                                       long long HW, long long total, int per_pixel) {
  long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= total) return;
  const long long b = pix / HW, p = pix - b * HW;
  const float* pp = prob + b * D * HW + p;
  const float* hp = per_pixel ? hyp + b * D * HW + p : hyp + b * D;
  const long long hs = per_pixel ? HW : 1;
  const float dep = depth[pix];
  const float gd = g_depth ? g_depth[pix] : 0.f;
  float gv = g_var ? g_var[pix] : 0.f;
  // S = sum p (d - depth)^2, var = 3 sqrt(S): d var / d p_k = 3/(2 sqrt S) (d_k - depth)^2 (the cross term vanishes)
  float S = 0.f;
  if (gv != 0.f) {
    for (int k = 0; k < D; ++k) {
      const float t = __ldg(hp + k * hs) - dep;
      S += __ldg(pp + (long long)k * HW) * t * t;
    }
  }
  const float cv = (gv != 0.f && S > 0.f) ? gv * 1.5f * rsqrtf(S) : 0.f;
  const float* gp = g_prob ? g_prob + b * D * HW + p : nullptr;
  float dot = 0.f;  // sum_j p_j g_p[j]
  for (int k = 0; k < D; ++k) {
    const float dk = __ldg(hp + k * hs), t = dk - dep;
    const float g = gd * dk + cv * t * t + (gp ? __ldg(gp + (long long)k * HW) : 0.f);
    dot += __ldg(pp + (long long)k * HW) * g;
  }
  float* gl = g_logits + b * D * HW + p;
  float* gh = (g_hyp && per_pixel) ? g_hyp + b * D * HW + p : nullptr;
  for (int k = 0; k < D; ++k) {
    const float dk = __ldg(hp + k * hs), t = dk - dep, pk = __ldg(pp + (long long)k * HW);
    const float g = gd * dk + cv * t * t + (gp ? __ldg(gp + (long long)k * HW) : 0.f);
    gl[(long long)k * HW] = pk * (g - dot);
    if (gh) gh[(long long)k * HW] = gd * pk + 2.f * cv * pk * t;
  }
}

// ---------------------------------------------------------------------------------------------
// dW for one (tap, ci-group, co-group): 64 accumulators per thread over a strided set of output voxels.
struct WgradParams {
  const void* x;    // G8 [B][Gin][Din][Hin][Win][8]
  const void* gy;   // G8 [B][Gout][Dout][Hout][Wout][8]
  float* dw;        // PyTorch layout: conv [Cout][Cin][27], transposed [Cin][Cout][27]
  int B, Cin, Cout, Din, Hin, Win, Dout, Hout, Wout, stride, transposed;
};

template <typename TX, typename TG>
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const WgradParams P) {
  const int Gin = P.Cin / 8, Gout = (P.Cout + 7) / 8;
  int combo = blockIdx.y;
  const int cog = combo % Gout; combo /= Gout;
  const int cig = combo % Gin; combo /= Gin;
  const int tap = combo;  // 0..26
  const int kd = tap / 9, kh = (tap / 3) % 3, kw = tap % 3;
  const long long HWo = (long long)P.Hout * P.Wout, Vo = HWo * P.Dout, total = Vo * P.B;
  float acc[8][8];  // [co][ci]
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[a][c] = 0.f;
  const TX* x = reinterpret_cast<const TX*>(P.x);
  const TG* gy = reinterpret_cast<const TG*>(P.gy);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / Vo);
    const long long r = idx - (long long)b * Vo;
    const int z = (int)(r / HWo);
    const int rem = (int)(r - (long long)z * HWo);
    const int y = rem / P.Wout, xx = rem - y * P.Wout;
    int zi, yi, xi;
    if (P.transposed) {  // o = 2 i - 1 + t
      int n = z + 1 - kd; if (n & 1) continue; zi = n >> 1;
      n = y + 1 - kh; if (n & 1) continue; yi = n >> 1;
      n = xx + 1 - kw; if (n & 1) continue; xi = n >> 1;
    } else {
      zi = z * P.stride - 1 + kd; yi = y * P.stride - 1 + kh; xi = xx * P.stride - 1 + kw;
    }
    if (zi < 0 || zi >= P.Din || yi < 0 || yi >= P.Hin || xi < 0 || xi >= P.Win) continue;
    const F8 g = load8(gy + g8_offset(b, cog, z, y, xx, Gout, P.Dout, P.Hout, P.Wout));
    const F8 v = load8(x + g8_offset(b, cig, zi, yi, xi, Gin, P.Din, P.Hin, P.Win));
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[a][c] = fmaf(g.v[a], v.v[c], acc[a][c]);
  }
  // block reduction: warp shuffles, then one atomic per (co, ci) per warp
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float s = acc[a][c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0 && s != 0.f) {
        const int co = cog * 8 + a, ci = cig * 8 + c;
        if (co < P.Cout) {
          float* dst = P.transposed ? P.dw + ((size_t)ci * P.Cout + co) * 27 + tap : P.dw + ((size_t)co * P.Cin + ci) * 27 + tap;
          atomicAdd(dst, s);
        }
      }
    }
}

int conv_wgrad_mma_launch(const damvs_conv3d_desc* d, const void* x, const void* g_y, float* dw, cudaStream_t st);   // wgrad_mma.cu

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_softmax_regress_bwd(const float* prob, const float* depth_hyp, const float* depth,
                                         const float* g_depth, const float* g_var, const float* g_prob, float* g_logits,
                                         float* g_hyp, int B, int D, int H, int W, int per_pixel_hyp, void* stream) {
  DAMVS_REQUIRE(prob && depth_hyp && depth && g_logits, "softmax_regress_bwd: null pointer");
  DAMVS_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0, "softmax_regress_bwd: bad shape");
  const long long HW = (long long)H * W, total = HW * B;
  head_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(prob, depth_hyp, depth, g_depth, g_var, g_prob,
                                                                                      g_logits, g_hyp, D, HW, total, per_pixel_hyp);
  DAMVS_LAUNCH_OK("head_bwd kernel");
  return DAMVS_OK;
}

extern "C" int damvs_conv3d_wgrad(const damvs_conv3d_desc* d, const void* x, const void* g_y, float* dw, void* stream) {
  DAMVS_REQUIRE(d && x && g_y && dw, "conv3d_wgrad: null pointer");
  DAMVS_REQUIRE(d->Cin > 0 && d->Cin % 8 == 0 && d->Cout > 0, "conv3d_wgrad: bad channels");
  DAMVS_REQUIRE(d->transposed || d->stride == 1 || d->stride == 2, "conv3d_wgrad: bad stride");
  WgradParams P;
  P.x = x; P.gy = g_y; P.dw = dw;
  P.B = d->B; P.Cin = d->Cin; P.Cout = d->Cout; P.Din = d->Din; P.Hin = d->Hin; P.Win = d->Win;
  P.stride = d->stride; P.transposed = d->transposed;
  if (d->transposed) { P.Dout = 2 * d->Din; P.Hout = 2 * d->Hin; P.Wout = 2 * d->Win; }
  else { P.Dout = (d->Din - 1) / d->stride + 1; P.Hout = (d->Hin - 1) / d->stride + 1; P.Wout = (d->Win - 1) / d->stride + 1; }
  const int Gin = d->Cin / 8, Gout = (d->Cout + 7) / 8;
  const long long total = (long long)P.B * P.Dout * P.Hout * P.Wout;
  int bx = (int)std::min<long long>((total + 255) / 256, 148 * 4 / std::max(1, std::min(4, Gin * Gout)) + 1);
  if (bx < 1) bx = 1;
  dim3 grid(bx, 27 * Gin * Gout);
  cudaStream_t st = (cudaStream_t)stream;
  DAMVS_CUDA_OK(cudaMemsetAsync(dw, 0, (size_t)d->Cin * d->Cout * 27 * sizeof(float), st));
  {
    // bf16 volumes: tensor-core kernel (wgrad_mma.cu); everything else: the fp32 CUDA-core kernel below
    const int rc = conv_wgrad_mma_launch(d, x, g_y, dw, st);
    if (rc != DAMVS_ERR_UNSUPPORTED) return rc;
  }
  const bool xf = d->in_dtype == DAMVS_F32, gf = d->out_dtype == DAMVS_F32;
  if (xf && gf) conv_wgrad_kernel<float, float><<<grid, 256, 0, st>>>(P);
  else if (!xf && !gf) conv_wgrad_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>(P);
  else if (xf) conv_wgrad_kernel<float, __nv_bfloat16><<<grid, 256, 0, st>>>(P);
  else conv_wgrad_kernel<__nv_bfloat16, float><<<grid, 256, 0, st>>>(P);
  DAMVS_LAUNCH_OK("conv_wgrad kernel");
  return DAMVS_OK;
}
