// Softmax / depth-regression / photometric-confidence / variance head.
//
// Replaces reference models/cas_mvsnet.py:105-124 and depth_regression
// (models/module.py:609-615): one pass over the logits and hypotheses, one
// store of the probability volume and three [B,H,W] maps.  HBM-bound streaming:
// algorithmic bytes per pixel = 2*D*4 read + D*4 + 12 written.
//
// Mapping: one thread per pixel; lanes run along W so every load/store of plane
// k is a coalesced 128-byte line per warp.  A pixel's column is strided by H*W
// in memory; the main kernel stages a D x 128-pixel tile in shared memory with
// cp.async, a streaming kernel covers any D / alignment.

#include "common.cuh"

namespace damvs {

// Staged variant (D <= 64, H*W % 4 == 0): a CTA owns 128 consecutive pixels; the D x 128 logits and
// hypotheses tiles are pulled into shared memory with 16-byte cp.async (no registers held while the loads
// are in flight, so many CTAs per SM keep HBM busy), then every thread walks its own column in shared
// memory (bank = pixel, conflict free) for max, sum, probabilities, regression, confidence and variance.
constexpr int kHeadPix = 128;

// exp(x) for x = logit - max <= 0 with the argument clamped at -80.  Peaked probability volumes (what a trained net -- or
// the synthetic benchmark net -- produces) put most hypotheses hundreds of units below the maximum: expf then returns
// denormals, and both expf and the IEEE division p = e / s drop into their slow paths (ncu, stage 2 of the benchmark:
// 162 warp instructions per (warp, hypothesis), 111 us for 182 MB).  exp(-80) = 1.8e-35 keeps e and e / s (s <= D) in the
// normal range; the probabilities it replaces are < 1.8e-35 in the reference too, far below one fp32 ulp of any output.
// The clamp is a compare, not fmaxf: fmaxf(NaN, -80) is -80, which would turn a NaN logit into a finite probability
// and hide a diverged training step behind plausible depth / confidence / variance.
__device__ __forceinline__ float exp_clamped(float x) { return expf(x < -80.f ? -80.f : x); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}

__global__ void __launch_bounds__(kHeadPix) head_staged_kernel(const float* __restrict__ logits,
                                                               const float* __restrict__ hyp, float* __restrict__ prob,
                                                               float* __restrict__ depth, float* __restrict__ conf,
                                                               float* __restrict__ var, int D, long long HW,
                                                               int per_pixel) {
  extern __shared__ __align__(16) float sm[];  // [D][128] logits, then [D][128] hypotheses
  float* sl = sm;
  float* sh = sm + D * kHeadPix;
  const int b = blockIdx.y;
  const long long p0 = (long long)blockIdx.x * kHeadPix;
  const int np = (int)min((long long)kHeadPix, HW - p0);  // multiple of 4
  const int t = threadIdx.x;
  const float* lg = logits + (long long)b * D * HW + p0;
  const float* hg = hyp + (long long)b * D * HW + p0;
  // 32 threads cover one plane's 128 pixels with 16-byte copies; 4 planes per sweep
  const int seg = (t & 31) * 4, kofs = t >> 5;
  if (seg < np) {
    for (int k = kofs; k < D; k += 4) {
      cp_async16(sl + k * kHeadPix + seg, lg + (long long)k * HW + seg);
      if (per_pixel) cp_async16(sh + k * kHeadPix + seg, hg + (long long)k * HW + seg);
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if (t >= np) return;
  const float* hb = hyp + (long long)b * D;  // [B,D] hypotheses
  float m = -INFINITY;
  for (int k = 0; k < D; ++k) m = fmaxf(m, sl[k * kHeadPix + t]);
  float s = 0.f;
  for (int k = 0; k < D; ++k) {
    const float e = exp_clamped(sl[k * kHeadPix + t] - m);
    sl[k * kHeadPix + t] = e;
    s += e;
  }
  float dsum = 0.f, isum = 0.f;
  float* pr = prob ? prob + (long long)b * D * HW + p0 + t : nullptr;
  const float inv_s = 1.f / s;   // one IEEE division per pixel; p = e * (1 / s) (see head_reg_kernel)
  for (int k = 0; k < D; ++k) {
    const float pk = sl[k * kHeadPix + t] * inv_s;
    sl[k * kHeadPix + t] = pk;
    const float dk = per_pixel ? sh[k * kHeadPix + t] : __ldg(hb + k);
    dsum += pk * dk;
    isum += pk * (float)k;
    if (pr) __stcs(pr + (long long)k * HW, pk);
  }
  float d2sum = 0.f;
  for (int k = 0; k < D; ++k) {
    const float dk = per_pixel ? sh[k * kHeadPix + t] : __ldg(hb + k);
    const float df = dk - dsum;
    d2sum += (df * df) * sl[k * kHeadPix + t];
  }
  long long idx = (long long)isum;  // .long() truncation, reference cas_mvsnet.py:116
  idx = idx < 0 ? 0 : (idx > D - 1 ? D - 1 : idx);
  float c = 0.f;
  for (int k = (int)idx - 1; k <= (int)idx + 2; ++k)
    if (k >= 0 && k < D) c += sl[k * kHeadPix + t];
  const long long o = (long long)b * HW + p0 + t;
  depth[o] = dsum;
  conf[o] = c;
  var[o] = 3.f * sqrtf(d2sum);
}

// Register variant (D in {8, 16, 32, 48, 64, 96}, per-pixel hypotheses): one thread per pixel holds its whole logits column
// in registers.  All D loads of a column are independent and issued back to back (D x 128-byte lines in flight per warp),
// the hypothesis column follows the same way while the soft-max runs, and nothing waits on a CTA-wide barrier: measured
// in situ (DRAM-cold inputs, right after the `prob` convolution) the staged kernel above spent most of its time with
// every warp of a CTA parked behind one cp.async group + __syncthreads (108 us for the 182 MB of stage 2 = 1.7 TB/s).
// Arithmetic is the staged kernel's (expf, one IEEE reciprocal per pixel, the reference's operation order), so the two
// kernels give bit-identical results.
template <int D>
__global__ void __launch_bounds__(128) head_reg_kernel(const float* __restrict__ logits, const float* __restrict__ hyp,
                                                       float* __restrict__ prob, float* __restrict__ depth, float* __restrict__ conf,
                                                       float* __restrict__ var, long long HW) {
  const int b = blockIdx.y;
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float* lg = logits + (long long)b * D * HW + p;
  const float* hg = hyp + (long long)b * D * HW + p;
  float e[D], h[D];
#pragma unroll
  for (int k = 0; k < D; ++k) e[k] = __ldcs(lg + (long long)k * HW);
#pragma unroll
  for (int k = 0; k < D; ++k) h[k] = __ldcs(hg + (long long)k * HW);
  float m = -INFINITY;
#pragma unroll
  for (int k = 0; k < D; ++k) m = fmaxf(m, e[k]);
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    e[k] = exp_clamped(e[k] - m);
    s += e[k];
  }
  float dsum = 0.f, isum = 0.f;
  float* pr = prob ? prob + (long long)b * D * HW + p : nullptr;
  // One IEEE division per pixel, then p = e * (1 / s): D divisions per pixel (FCHK + ~10 instructions each, plus the
  // slow-path call) were a third of this kernel's instructions and kept stage 2 issue-bound (ncu: 92 warp instructions
  // per hypothesis, issue slots 64 % busy, 2.9 TB/s).  The product differs from the quotient by at most one ulp.
  const float inv_s = 1.f / s;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const float pk = e[k] * inv_s;
    e[k] = pk;
    dsum += pk * h[k];
    isum += pk * (float)k;
    if (pr) __stcs(pr + (long long)k * HW, pk);
  }
  float d2sum = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const float df = h[k] - dsum;
    d2sum += (df * df) * e[k];
  }
  long long idx = (long long)isum;  // .long() truncation, reference cas_mvsnet.py:116
  idx = idx < 0 ? 0 : (idx > D - 1 ? D - 1 : idx);
  const int i0 = (int)idx - 1, i1 = (int)idx + 2;
  float c = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) c += (k >= i0 && k <= i1) ? e[k] : 0.f;   // same ascending order as the staged kernel's window loop
  const long long o = (long long)b * HW + p;
  depth[o] = dsum;
  conf[o] = c;
  var[o] = 3.f * sqrtf(d2sum);
}

// Any D: three passes over the logits column (re-reads are L2 hits).
__global__ void __launch_bounds__(256) head_stream_kernel(const float* __restrict__ logits,
                                                          const float* __restrict__ hyp, float* __restrict__ prob,
                                                          float* __restrict__ depth, float* __restrict__ conf,
                                                          float* __restrict__ var, int D, long long HW,
                                                          long long total, int per_pixel) {
  long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= total) return;
  long long b = pix / HW;
  long long p = pix - b * HW;
  const float* lg = logits + b * D * HW + p;
  const float* hp = per_pixel ? hyp + b * D * HW + p : hyp + b * D;
  const long long hs = per_pixel ? HW : 1;
  float m = -INFINITY;
  for (int k = 0; k < D; ++k) m = fmaxf(m, __ldg(lg + (long long)k * HW));
  float s = 0.f;
  for (int k = 0; k < D; ++k) s += exp_clamped(__ldg(lg + (long long)k * HW) - m);
  float dsum = 0.f, isum = 0.f;
  float* pr = prob ? prob + b * D * HW + p : nullptr;
  const float inv_s = 1.f / s;
  for (int k = 0; k < D; ++k) {
    float pk = exp_clamped(__ldg(lg + (long long)k * HW) - m) * inv_s;
    dsum += pk * __ldg(hp + k * hs);
    isum += pk * (float)k;
    if (pr) pr[(long long)k * HW] = pk;
  }
  long long idx = (long long)isum;
  idx = idx < 0 ? 0 : (idx > D - 1 ? D - 1 : idx);
  float d2sum = 0.f, c = 0.f;
  for (int k = 0; k < D; ++k) {
    float pk = exp_clamped(__ldg(lg + (long long)k * HW) - m) * inv_s;
    float t = __ldg(hp + k * hs) - dsum;
    d2sum += (t * t) * pk;
    if (k >= idx - 1 && k <= idx + 2) c += pk;
  }
  depth[pix] = dsum;
  conf[pix] = c;
  var[pix] = 3.f * sqrtf(d2sum);
}

__global__ void __launch_bounds__(256) depth_regression_kernel(const float* __restrict__ prob,
                                                               const float* __restrict__ hyp,
                                                               float* __restrict__ out, int D, long long HW,
                                                               long long total, int per_pixel) {
  long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= total) return;
  long long b = pix / HW;
  long long p = pix - b * HW;
  const float* pp = prob + b * D * HW + p;
  const float* hp = per_pixel ? hyp + b * D * HW + p : hyp + b * D;
  const long long hs = per_pixel ? HW : 1;
  float acc = 0.f;
  for (int k = 0; k < D; ++k) acc += __ldg(pp + (long long)k * HW) * __ldg(hp + k * hs);
  out[pix] = acc;
}

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_softmax_regress_fwd(const float* logits, const float* depth_hyp, float* prob, float* depth,
                                         float* conf, float* var, int B, int D, int H, int W, int per_pixel_hyp,
                                         void* stream) {
  DAMVS_REQUIRE(logits && depth_hyp && depth && conf && var, "softmax_regress: null pointer");
  DAMVS_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0, "softmax_regress: bad shape B=%d D=%d H=%d W=%d", B, D, H, W);
  long long HW = (long long)H * W, total = HW * B;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned blocks = (unsigned)((total + 255) / 256);
  const bool aligned = (HW % 4 == 0) && aligned16(logits) && aligned16(depth_hyp) && B <= 65535;
  if (per_pixel_hyp && B <= 65535 && (D == 8 || D == 16 || D == 32 || D == 48 || D == 64 || D == 96)) {
    // small maps (stage 1: 115 k pixels) get 64-thread CTAs: twice the CTAs to spread over the 148 SMs
    const int threads = total < 148ll * 8 * 128 ? 64 : 128;
    dim3 grid((unsigned)((HW + threads - 1) / threads), B);
#define GO(DD) head_reg_kernel<DD><<<grid, threads, 0, st>>>(logits, depth_hyp, prob, depth, conf, var, HW)
    if (D == 8) GO(8); else if (D == 16) GO(16); else if (D == 32) GO(32); else if (D == 48) GO(48); else if (D == 64) GO(64); else GO(96);
#undef GO
  } else if (D <= 64 && aligned) {
    const size_t smem = (size_t)2 * D * kHeadPix * sizeof(float);
    if (smem > 48 * 1024)
      DAMVS_CUDA_OK(cudaFuncSetAttribute(head_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)((HW + kHeadPix - 1) / kHeadPix), B);
    head_staged_kernel<<<grid, kHeadPix, smem, st>>>(logits, depth_hyp, prob, depth, conf, var, D, HW, per_pixel_hyp);
  } else {
    head_stream_kernel<<<blocks, 256, 0, st>>>(logits, depth_hyp, prob, depth, conf, var, D, HW, total,
                                               per_pixel_hyp);
  }
  DAMVS_LAUNCH_OK("head kernel");
  return DAMVS_OK;
}

extern "C" int damvs_depth_regression_fwd(const float* prob, const float* depth_hyp, float* out, int B, int D,
                                          int H, int W, int per_pixel_hyp, void* stream) {
  DAMVS_REQUIRE(prob && depth_hyp && out, "depth_regression: null pointer");
  DAMVS_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0, "depth_regression: bad shape");
  long long HW = (long long)H * W, total = HW * B;
  unsigned blocks = (unsigned)((total + 255) / 256);
  depth_regression_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(prob, depth_hyp, out, D, HW, total,
                                                                     per_pixel_hyp);
  DAMVS_LAUNCH_OK("depth_regression kernel");
  return DAMVS_OK;
}
