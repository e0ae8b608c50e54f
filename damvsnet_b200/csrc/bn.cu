// Training-mode BatchNorm3d around the conv blocks of CostRegNet (reference models/module.py:141-159, 184-202:
// nn.BatchNorm3d(momentum=0.1) -> F.relu, with the skip adds of CostRegNet.forward, models/module.py:537-539).
//
// In training the convolution kernels write the raw conv output y; the batch statistics, the normalise + ReLU
// (+ skip) pass and the backward of that pass are the HBM-streaming kernels below.  All of them work on G8
// volumes [B][C/8][D][H][W][8] (bf16 or fp32), one thread per (voxel, 8-channel group), 16/32-byte accesses.
//
//   bn_stats_kernel    sums[c] += {sum y, sum y^2} over (B,D,H,W)        (fp32 partials around a pivot, fp64 atomics)
//   bn_apply_kernel    out = skip + act(y * scale[c] + shift[c])
//   bn_bwd_kernel      g_z = g_out * [act active];  sums[c] += {sum g_z, sum g_z*y};
//                      g_y = k1[c] * g_z + k2[c] * y + k3[c]
//   bn_finalize_kernel / bn_bwd_coeffs_kernel   the C-sized coefficient algebra between them (mean/var -> scale/shift
//                      and running buffers; BatchNorm backward formula -> k1,k2,k3, d gamma, d beta), one launch each.
#include "common.cuh"

namespace damvs {

constexpr int kStatVox = 16;  // voxels per thread in the reductions

template <typename T>
__global__ void __launch_bounds__(256) bn_stats_kernel(const T* __restrict__ y, double* __restrict__ sums, int G, long long V) {
  __shared__ float s_part[8][8][2];
  const int bg = blockIdx.y, g = bg % G;
  const long long v0 = ((long long)blockIdx.x * blockDim.x) * kStatVox + threadIdx.x;
  float a[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = q[j] = 0.f;
  const T* base = y + (size_t)bg * V * 8;
  // fp32 partials of (y - p) around a per-block pivot p (the block's first voxel), un-shifted in fp64: raw fp32 sums of
  // y and y^2 lose the variance to cancellation once |mean| >> std (relative error ~ (mean/std)^2 * 2^-24)
  const long long vb = (long long)blockIdx.x * blockDim.x * kStatVox;
  const F8 pv = load8(base + vb * 8);
#pragma unroll 4
  for (int k = 0; k < kStatVox; ++k) {
    const long long v = v0 + (long long)k * blockDim.x;
    if (v < V) {
      const F8 r = load8(base + v * 8);
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float d = r.v[j] - pv.v[j]; a[j] += d; q[j] = fmaf(d, d, q[j]); }
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a[j] += __shfl_xor_sync(0xffffffffu, a[j], o);
      q[j] += __shfl_xor_sync(0xffffffffu, q[j], o);
    }
    if (lane == 0) { s_part[warp][j][0] = a[j]; s_part[warp][j][1] = q[j]; }
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    const int j = threadIdx.x;
    double s1 = 0.0, s2 = 0.0;
    for (int k = 0; k < 8; ++k) { s1 += (double)s_part[k][j][0]; s2 += (double)s_part[k][j][1]; }
    const double p = pv.v[j], n = (double)min((long long)blockDim.x * kStatVox, V - vb);
    atomicAdd(sums + (g * 8 + j) * 2, s1 + n * p);
    atomicAdd(sums + (g * 8 + j) * 2 + 1, s2 + p * (2.0 * s1 + n * p));
  }
}

template <typename T>
__global__ void __launch_bounds__(256) bn_apply_kernel(const T* __restrict__ y, const float* __restrict__ scale,
                                                       const float* __restrict__ shift, const T* __restrict__ skip,
                                                       T* __restrict__ out, int G, long long V, int relu) {
  const int bg = blockIdx.y, g = bg % G;
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const size_t off = ((size_t)bg * V + v) * 8;
  F8 r = load8(y + off);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float z = fmaf(r.v[j], __ldg(scale + g * 8 + j), __ldg(shift + g * 8 + j));
    r.v[j] = relu ? fmaxf(z, 0.f) : z;
  }
  if (skip) {
    const F8 s = load8(skip + off);
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] += s.v[j];
  }
  store8(out + off, r);
}

template <typename T>
__global__ void __launch_bounds__(256) bn_bwd_kernel(const T* __restrict__ g_out, const T* __restrict__ y,
                                                     const float* __restrict__ scale, const float* __restrict__ shift,
                                                     const float* __restrict__ k1, const float* __restrict__ k2,
                                                     const float* __restrict__ k3, T* __restrict__ g_y,
                                                     double* __restrict__ sums, int G, long long V, int relu) {
  __shared__ float s_part[8][8][2];
  const int bg = blockIdx.y, g = bg % G;
  const long long v0 = ((long long)blockIdx.x * blockDim.x) * kStatVox + threadIdx.x;
  float a[8], q[8], sc[8], sh[8], c1[8], c2[8], c3[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    a[j] = q[j] = 0.f;
    sc[j] = scale ? __ldg(scale + g * 8 + j) : 1.f;
    sh[j] = shift ? __ldg(shift + g * 8 + j) : 0.f;
    c1[j] = k1 ? __ldg(k1 + g * 8 + j) : 1.f;
    c2[j] = k2 ? __ldg(k2 + g * 8 + j) : 0.f;
    c3[j] = k3 ? __ldg(k3 + g * 8 + j) : 0.f;
  }
  const size_t base = (size_t)bg * V * 8;
  // sum g_z * y accumulated as sum g_z * (y - p) + p * sum g_z (pivot p as in bn_stats_kernel), so that the backward's
  // sum g_z y - mean * sum g_z cancels in fp64 rather than in the fp32 partials
  float pv[8];
  {
    const F8 r = load8(y + base + (size_t)blockIdx.x * blockDim.x * kStatVox * 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) pv[j] = r.v[j];
  }
#pragma unroll 2
  for (int k = 0; k < kStatVox; ++k) {
    const long long v = v0 + (long long)k * blockDim.x;
    if (v < V) {
      const size_t off = base + v * 8;
      const F8 go = load8(g_out + off), yy = load8(y + off);
      F8 r;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool on = !relu || fmaf(yy.v[j], sc[j], sh[j]) > 0.f;
        const float gz = on ? go.v[j] : 0.f;
        a[j] += gz;
        q[j] = fmaf(gz, yy.v[j] - pv[j], q[j]);
        r.v[j] = fmaf(c1[j], gz, fmaf(c2[j], yy.v[j], c3[j]));
      }
      if (g_y) store8(g_y + off, r);
    }
  }
  if (sums) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a[j] += __shfl_xor_sync(0xffffffffu, a[j], o);
        q[j] += __shfl_xor_sync(0xffffffffu, q[j], o);
      }
      if (lane == 0) { s_part[warp][j][0] = a[j]; s_part[warp][j][1] = q[j]; }
    }
    __syncthreads();
    if (threadIdx.x < 8) {
      const int j = threadIdx.x;
      double s1 = 0.0, s2 = 0.0;
      for (int k = 0; k < 8; ++k) { s1 += (double)s_part[k][j][0]; s2 += (double)s_part[k][j][1]; }
      atomicAdd(sums + (g * 8 + j) * 2, s1);
      atomicAdd(sums + (g * 8 + j) * 2 + 1, s2 + (double)pv[j] * s1);
    }
  }
}

// [B][D][H][W] fp32 -> G8 volume with one group: channel 0 = value, channels 1..7 = 0
template <typename T>
__global__ void __launch_bounds__(256) plain_to_g8_kernel(const float* __restrict__ in, T* __restrict__ out, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  F8 r;
  r.v[0] = __ldg(in + i);
#pragma unroll
  for (int j = 1; j < 8; ++j) r.v[j] = 0.f;
  store8(out + i * 8, r);
}

// C-sized coefficient algebra of a training-mode BatchNorm, one thread per channel (replaces ~12 tiny tensor ops per block).
// Forward: batch mean / biased variance from the fp64 sums, running-buffer update (momentum, unbiased variance), and the
// folded affine scale = gamma * rstd, shift = beta - mean * scale.
__global__ void bn_finalize_kernel(const double* __restrict__ sums, const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* __restrict__ running_mean, float* __restrict__ running_var, double count, float momentum, float eps,
                                   float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                   int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = sums[2 * c] / count;
  double var = sums[2 * c + 1] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  if (running_mean) {
    running_mean[c] = (float)((1.0 - momentum) * (double)running_mean[c] + momentum * mean);
    running_var[c] = (float)((1.0 - momentum) * (double)running_var[c] + momentum * var * (count / fmax(count - 1.0, 1.0)));
  }
  const double rstd = rsqrt(var + (double)eps);
  const double g = gamma ? (double)gamma[c] : 1.0, b = beta ? (double)beta[c] : 0.0;
  const double sc = g * rstd;
  scale[c] = (float)sc;
  shift[c] = (float)(b - mean * sc);
  mean_out[c] = (float)mean;
  rstd_out[c] = (float)rstd;
}

// Backward: from sums = {sum g_z, sum g_z * y}:  d gamma = rstd (sum g_z y - mean sum g_z),  d beta = sum g_z, and (batch
// statistics only) the coefficients of g_y = k1 g_z + k2 y + k3 = scale (g_z - mean(g_z) - yhat mean(g_z yhat)).
__global__ void bn_bwd_coeffs_kernel(const double* __restrict__ sums, const float* __restrict__ scale, const float* __restrict__ mean,
                                     const float* __restrict__ rstd, double count, float* __restrict__ k1, float* __restrict__ k2,
                                     float* __restrict__ k3, float* __restrict__ g_gamma, float* __restrict__ g_beta, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double sg = sums[2 * c], sgy = sums[2 * c + 1], mu = mean[c], rs = rstd[c], sc = scale[c];
  const double dot = rs * (sgy - mu * sg);
  if (g_gamma) g_gamma[c] = (float)dot;
  if (g_beta) g_beta[c] = (float)sg;
  if (k1) {
    const double m1 = sg / count, m2 = dot / count;
    k1[c] = (float)sc;
    k2[c] = (float)(-sc * rs * m2);
    k3[c] = (float)(sc * (mu * rs * m2 - m1));
  }
}

static bool vol_args_ok(int B, int C, int D, int H, int W) {
  return B > 0 && C > 0 && C % 8 == 0 && D > 0 && H > 0 && W > 0 && (long long)B * (C / 8) <= 65535;
}

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_bn_stats(const void* y, int dtype, int B, int C, int D, int H, int W, double* sums, void* stream) {
  DAMVS_REQUIRE(y && sums, "bn_stats: null pointer");
  DAMVS_REQUIRE(vol_args_ok(B, C, D, H, W), "bn_stats: bad shape");
  DAMVS_REQUIRE(aligned16(y), "bn_stats: y must be 16-byte aligned");
  const long long V = (long long)D * H * W;
  const int G = C / 8;
  dim3 grid((unsigned)((V + 256 * kStatVox - 1) / (256 * kStatVox)), B * G);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DAMVS_F32) bn_stats_kernel<float><<<grid, 256, 0, st>>>((const float*)y, sums, G, V);
  else if (dtype == DAMVS_BF16) bn_stats_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)y, sums, G, V);
  else return set_error(DAMVS_ERR_INVALID, "bn_stats: bad dtype %d", dtype);
  DAMVS_LAUNCH_OK("bn_stats kernel");
  return DAMVS_OK;
}

extern "C" int damvs_bn_apply(const void* y, const float* scale, const float* shift, const void* skip, void* out, int dtype,
                              int B, int C, int D, int H, int W, int relu, void* stream) {
  DAMVS_REQUIRE(y && scale && shift && out, "bn_apply: null pointer");
  DAMVS_REQUIRE(vol_args_ok(B, C, D, H, W), "bn_apply: bad shape");
  DAMVS_REQUIRE(aligned16(y) && aligned16(out) && aligned16(skip), "bn_apply: pointers must be 16-byte aligned");
  const long long V = (long long)D * H * W;
  const int G = C / 8;
  dim3 grid((unsigned)((V + 255) / 256), B * G);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DAMVS_F32)
    bn_apply_kernel<float><<<grid, 256, 0, st>>>((const float*)y, scale, shift, (const float*)skip, (float*)out, G, V, relu);
  else if (dtype == DAMVS_BF16)
    bn_apply_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)y, scale, shift, (const __nv_bfloat16*)skip,
                                                        (__nv_bfloat16*)out, G, V, relu);
  else return set_error(DAMVS_ERR_INVALID, "bn_apply: bad dtype %d", dtype);
  DAMVS_LAUNCH_OK("bn_apply kernel");
  return DAMVS_OK;
}

extern "C" int damvs_bn_bwd(const void* g_out, const void* y, const float* scale, const float* shift, const float* k1,
                            const float* k2, const float* k3, void* g_y, double* sums, int dtype, int B, int C, int D, int H,
                            int W, int relu, void* stream) {
  DAMVS_REQUIRE(g_out && y && (g_y || sums), "bn_bwd: null pointer");
  DAMVS_REQUIRE(vol_args_ok(B, C, D, H, W), "bn_bwd: bad shape");
  DAMVS_REQUIRE(aligned16(g_out) && aligned16(y) && aligned16(g_y), "bn_bwd: pointers must be 16-byte aligned");
  const long long V = (long long)D * H * W;
  const int G = C / 8;
  dim3 grid((unsigned)((V + 256 * kStatVox - 1) / (256 * kStatVox)), B * G);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DAMVS_F32)
    bn_bwd_kernel<float><<<grid, 256, 0, st>>>((const float*)g_out, (const float*)y, scale, shift, k1, k2, k3, (float*)g_y, sums, G, V, relu);
  else if (dtype == DAMVS_BF16)
    bn_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)g_out, (const __nv_bfloat16*)y, scale, shift, k1, k2, k3,
                                                      (__nv_bfloat16*)g_y, sums, G, V, relu);
  else return set_error(DAMVS_ERR_INVALID, "bn_bwd: bad dtype %d", dtype);
  DAMVS_LAUNCH_OK("bn_bwd kernel");
  return DAMVS_OK;
}

extern "C" int damvs_bn_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                                 double count, float momentum, float eps, float* scale, float* shift, float* mean, float* rstd, int C,
                                 void* stream) {
  DAMVS_REQUIRE(sums && scale && shift && mean && rstd && C > 0 && count > 0, "bn_finalize: bad arguments");
  DAMVS_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "bn_finalize: running buffers come in pairs");
  bn_finalize_kernel<<<(C + 63) / 64, 64, 0, (cudaStream_t)stream>>>(sums, gamma, beta, running_mean, running_var, count, momentum, eps, scale,
                                                                   shift, mean, rstd, C);
  DAMVS_LAUNCH_OK("bn_finalize kernel");
  return DAMVS_OK;
}

extern "C" int damvs_bn_bwd_coeffs(const double* sums, const float* scale, const float* mean, const float* rstd, double count, float* k1,
                                   float* k2, float* k3, float* g_gamma, float* g_beta, int C, void* stream) {
  DAMVS_REQUIRE(sums && scale && mean && rstd && C > 0 && count > 0, "bn_bwd_coeffs: bad arguments");
  DAMVS_REQUIRE((k1 == nullptr) == (k2 == nullptr) && (k1 == nullptr) == (k3 == nullptr), "bn_bwd_coeffs: k1, k2, k3 come together");
  bn_bwd_coeffs_kernel<<<(C + 63) / 64, 64, 0, (cudaStream_t)stream>>>(sums, scale, mean, rstd, count, k1, k2, k3, g_gamma, g_beta, C);
  DAMVS_LAUNCH_OK("bn_bwd_coeffs kernel");
  return DAMVS_OK;
}

extern "C" int damvs_plain_to_g8(const float* in, void* out, int dtype, long long voxels, void* stream) {
  DAMVS_REQUIRE(in && out && voxels > 0, "plain_to_g8: bad arguments");
  DAMVS_REQUIRE(aligned16(out), "plain_to_g8: out must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned nb = (unsigned)((voxels + 255) / 256);
  if (dtype == DAMVS_F32) plain_to_g8_kernel<float><<<nb, 256, 0, st>>>(in, (float*)out, voxels);
  else if (dtype == DAMVS_BF16) plain_to_g8_kernel<__nv_bfloat16><<<nb, 256, 0, st>>>(in, (__nv_bfloat16*)out, voxels);
  else return set_error(DAMVS_ERR_INVALID, "plain_to_g8: bad dtype %d", dtype);
  DAMVS_LAUNCH_OK("plain_to_g8 kernel");
  return DAMVS_OK;
}
