// Direct (CUDA-core, fp32-accumulate) 3x3x3 convolution blocks of CostRegNet.
//
// This is the exact-arithmetic implementation of damvs_conv3d_fwd
// (impl = DAMVS_CONV_DIRECT): fp32 multiply-add in a fixed order, used for the
// "fp32 relative depth error <= 1e-4" parity claim and for layer shapes the
// tcgen05 implicit-GEMM kernel (conv3d_tc.cu) does not cover.  It replaces
// Conv3d / Deconv3d (reference models/module.py:117-202) with eval-mode
// BatchNorm folded into a per-channel affine, plus the skip-add of
// CostRegNet.forward (models/module.py:532-541).
//
// Mapping: a thread owns one output voxel and one group of 8 output channels;
// the 27*Cin*8 weights of that group sit in shared memory and are read as
// warp-wide broadcasts; input voxels are 8-channel vectors of the G8 volume.
#include <algorithm>

#include "common.cuh"

namespace damvs {

struct ConvParams {
  const void* in;
  const float* w;      // [Gout][27][Cin][8]
  const float* scale;  // [Cout] or null
  const float* shift;
  const void* skip;
  void* out;
  int B, Cin, Cout, Din, Hin, Win, Dout, Hout, Wout, stride, transposed, relu, plain_out;
};

// VX output voxels per thread, 32 apart along x (lane l of a warp owns x = strip * 32 * VX + v * 32 + l, v < VX): every
// weight vector read from shared memory feeds 8 * VX FMAs instead of 8 (the one-voxel version issued one LDS.128 per four
// FMAs and ran at 24 % of the fp32 peak), while the loads of one v stay coalesced across the warp (VX ADJACENT voxels per
// thread put the lanes 128 bytes apart and made it slower).  Each output's own arithmetic -- tap order (kd, kh, kw),
// channels in order inside a tap, two-level summation -- is unchanged: results are bit-identical to the one-voxel kernel.
// ONE = the `prob` layer (one output channel, plain fp32 output): only channel 0 of the zero-padded weight group is
// computed (the general path spent 7/8 of that layer's FMAs on the padding).
template <typename TIn, typename TOut, int kVX, bool ONE>
__global__ void __launch_bounds__(128) conv3d_direct_kernel(const ConvParams P) {
  extern __shared__ float s_w[];  // [27][Cin][8]
  const int g = blockIdx.y, b = blockIdx.z;
  const int Cin = P.Cin, Gin = Cin / 8;
  const int nw = 27 * Cin * 8;
  const float* wsrc = P.w + (size_t)g * nw;
  for (int i = threadIdx.x * 4; i < nw; i += blockDim.x * 4)
    *reinterpret_cast<float4*>(s_w + i) = __ldg(reinterpret_cast<const float4*>(wsrc + i));
  __syncthreads();

  // CTA = 4 warps = 4 consecutive output rows of one strip of 32 * VX voxels: the kh taps of a row are the rows its sibling
  // warps load, so they hit in L1 (one row per CTA left every tap but kw to L2)
  const int Ws = (P.Wout + 32 * kVX - 1) / (32 * kVX);     // strips per output row
  const int Hb = (P.Hout + 3) / 4;                          // row blocks
  const long long per_plane = (long long)Hb * Ws;
  const long long HWo = (long long)P.Hout * P.Wout;
  const long long Vo = HWo * P.Dout;
  const long long cid = blockIdx.x;                         // (z, row block, strip)
  const int z = (int)(cid / per_plane);
  const int rem = (int)(cid - (long long)z * per_plane);
  const int y = (rem / Ws) * 4 + (threadIdx.x >> 5);
  const int x0 = (rem % Ws) * (32 * kVX) + (threadIdx.x & 31);
  if (z >= P.Dout || y >= P.Hout) return;

  float acc[kVX][8];
#pragma unroll
  for (int v = 0; v < kVX; ++v)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[v][j] = 0.f;

  const TIn* in = reinterpret_cast<const TIn*>(P.in);
  for (int kd = 0; kd < 3; ++kd) {
    int zi;
    if (P.transposed) {
      int num = z + 1 - kd;  // o = 2i - 1 + t
      if (num & 1) continue;
      zi = num >> 1;
    } else {
      zi = z * P.stride - 1 + kd;
    }
    if (zi < 0 || zi >= P.Din) continue;
    for (int kh = 0; kh < 3; ++kh) {
      int yi;
      if (P.transposed) {
        int num = y + 1 - kh;
        if (num & 1) continue;
        yi = num >> 1;
      } else {
        yi = y * P.stride - 1 + kh;
      }
      if (yi < 0 || yi >= P.Hin) continue;
      for (int kw = 0; kw < 3; ++kw) {
        int xi[kVX];
        bool ok[kVX], any = false;
#pragma unroll
        for (int v = 0; v < kVX; ++v) {
          const int x = x0 + 32 * v;
          if (P.transposed) {
            const int num = x + 1 - kw;
            xi[v] = num >> 1;
            ok[v] = !(num & 1);
          } else {
            xi[v] = x * P.stride - 1 + kw;
            ok[v] = true;
          }
          ok[v] = ok[v] && x < P.Wout && xi[v] >= 0 && xi[v] < P.Win;
          any = any || ok[v];
        }
        if (!any) continue;
        const float* wt = s_w + ((kd * 3 + kh) * 3 + kw) * Cin * 8;
        // two-level summation: the Cin products of one tap go into a fresh partial, the <= 27 partials into acc.  The
        // rounding error grows with sqrt(Cin) + sqrt(27) instead of sqrt(27 * Cin) (up to 1728 terms).
        float part[kVX][8];
#pragma unroll
        for (int v = 0; v < kVX; ++v)
#pragma unroll
          for (int j = 0; j < 8; ++j) part[v][j] = 0.f;
        for (int gi = 0; gi < Gin; ++gi) {
          F8 val[kVX];
#pragma unroll
          for (int v = 0; v < kVX; ++v) {
            if (ok[v]) {
              val[v] = load8(in + g8_offset(b, gi, zi, yi, xi[v], Gin, P.Din, P.Hin, P.Win));
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) val[v].v[j] = 0.f;
            }
          }
#pragma unroll
          for (int ci = 0; ci < 8; ++ci) {
            if (ONE) {
              const float w0 = wt[(gi * 8 + ci) * 8];
#pragma unroll
              for (int v = 0; v < kVX; ++v) part[v][0] = fmaf(val[v].v[ci], w0, part[v][0]);
              continue;
            }
            const float4 wa = *reinterpret_cast<const float4*>(wt + (gi * 8 + ci) * 8);
            const float4 wb = *reinterpret_cast<const float4*>(wt + (gi * 8 + ci) * 8 + 4);
#pragma unroll
            for (int v = 0; v < kVX; ++v) {
              const float a = val[v].v[ci];
              part[v][0] = fmaf(a, wa.x, part[v][0]);
              part[v][1] = fmaf(a, wa.y, part[v][1]);
              part[v][2] = fmaf(a, wa.z, part[v][2]);
              part[v][3] = fmaf(a, wa.w, part[v][3]);
              part[v][4] = fmaf(a, wb.x, part[v][4]);
              part[v][5] = fmaf(a, wb.y, part[v][5]);
              part[v][6] = fmaf(a, wb.z, part[v][6]);
              part[v][7] = fmaf(a, wb.w, part[v][7]);
            }
          }
        }
#pragma unroll
        for (int v = 0; v < kVX; ++v)
          if (ok[v]) {           // a tap that does not exist for this voxel contributes nothing (not even +0: -0 stays -0)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[v][j] += part[v][j];
          }
      }
    }
  }

  const int Gout = P.Cout / 8;
#pragma unroll
  for (int v = 0; v < kVX; ++v) {
    const int x = x0 + 32 * v;
    if (x >= P.Wout) break;
    F8 r;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int co = g * 8 + j;
      float t = acc[v][j];
      if (P.scale && co < P.Cout) t = t * __ldg(P.scale + co) + __ldg(P.shift + co);
      if (P.relu) t = fmaxf(t, 0.f);
      r.v[j] = t;
    }
    if (P.plain_out) {
      reinterpret_cast<float*>(P.out)[(long long)b * Vo + (long long)z * HWo + (long long)y * P.Wout + x] = r.v[0];
      continue;
    }
    const size_t off = g8_offset(b, g, z, y, x, Gout, P.Dout, P.Hout, P.Wout);
    if (P.skip) {
      F8 sk = load8(reinterpret_cast<const TOut*>(P.skip) + off);
#pragma unroll
      for (int j = 0; j < 8; ++j) r.v[j] += sk.v[j];
    }
    store8(reinterpret_cast<TOut*>(P.out) + off, r);
  }
}

// PyTorch weight -> [Gout][27][Cin][8] fp32 (zero-padded to a multiple of 8 output channels)
__global__ void pack_weight_direct_kernel(const float* __restrict__ w, float* __restrict__ packed, int Cin, int Cout,
                                          int transposed, int total) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int j = i & 7;
  int ci = (i >> 3) % Cin;
  int t = (i / (8 * Cin)) % 27;
  int g = i / (8 * Cin * 27);
  int co = g * 8 + j;
  float v = 0.f;
  if (co < Cout) v = transposed ? w[((size_t)ci * Cout + co) * 27 + t] : w[((size_t)co * Cin + ci) * 27 + t];
  packed[i] = v;
}

int conv3d_direct_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, const float* scale,
                         const float* shift, const void* skip, void* out, cudaStream_t st) {
  ConvParams P;
  P.in = in; P.w = (const float*)packed; P.scale = scale; P.shift = shift; P.skip = skip; P.out = out;
  P.B = d->B; P.Cin = d->Cin; P.Cout = d->Cout; P.Din = d->Din; P.Hin = d->Hin; P.Win = d->Win;
  P.stride = d->stride; P.transposed = d->transposed; P.relu = d->relu; P.plain_out = d->plain_out;
  if (d->transposed) {
    P.Dout = 2 * d->Din; P.Hout = 2 * d->Hin; P.Wout = 2 * d->Win;
  } else {
    P.Dout = (d->Din - 1) / d->stride + 1; P.Hout = (d->Hin - 1) / d->stride + 1; P.Wout = (d->Win - 1) / d->stride + 1;
  }
  const int Gout = (d->Cout + 7) / 8;
  // voxels per thread (coarse levels are 50..100 wide); measured on B200 (fp32 pipeline at the DTU-test shape): 34.1 /
  // 43.0 / 41.7 views/s for 1 / 2 / 4 voxels per thread (4 costs occupancy: 128 registers), hence 2 wherever a row has
  // two 32-voxel strips
  const int vx = P.Wout >= 48 ? 2 : 1;
  const long long ctas = (long long)P.Dout * ((P.Hout + 3) / 4) * ((P.Wout + 32 * vx - 1) / (32 * vx));
  if (ctas > 0x7fffffffll) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d direct: volume too large for one launch");
  dim3 grid((unsigned)ctas, Gout, d->B);
  size_t smem = (size_t)27 * d->Cin * 8 * sizeof(float);
  if (smem > 200 * 1024) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d direct: Cin=%d too large", d->Cin);
#define LAUNCH_V(TI, TO, VX)                                                                                    \
  do {                                                                                                          \
    if (smem > 48 * 1024)                                                                                       \
      DAMVS_CUDA_OK(cudaFuncSetAttribute(conv3d_direct_kernel<TI, TO, VX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    if (one) conv3d_direct_kernel<TI, TO, VX, true><<<grid, 128, smem, st>>>(P);                                \
    else conv3d_direct_kernel<TI, TO, VX, false><<<grid, 128, smem, st>>>(P);                                   \
  } while (0)
#define LAUNCH(TI, TO)                                                                                          \
  do {                                                                                                          \
    if (vx == 2) LAUNCH_V(TI, TO, 2); else LAUNCH_V(TI, TO, 1);                                                 \
  } while (0)
  const bool out_f32 = d->plain_out || d->out_dtype == DAMVS_F32;
  const bool one = d->plain_out && smem <= 48 * 1024;   // Cout == 1 (checked by the C ABI); Cin <= 48 keeps the default smem limit
  const int od = out_f32 ? DAMVS_F32 : d->out_dtype;
  if (d->in_dtype == DAMVS_F32 && od == DAMVS_F32) LAUNCH(float, float);
  else if (d->in_dtype == DAMVS_F32 && od == DAMVS_BF16) LAUNCH(float, __nv_bfloat16);
  else if (d->in_dtype == DAMVS_F32 && od == DAMVS_F16) LAUNCH(float, __half);
  else if (d->in_dtype == DAMVS_BF16 && od == DAMVS_F32) LAUNCH(__nv_bfloat16, float);
  else if (d->in_dtype == DAMVS_BF16 && od == DAMVS_BF16) LAUNCH(__nv_bfloat16, __nv_bfloat16);
  else if (d->in_dtype == DAMVS_F16 && od == DAMVS_F32) LAUNCH(__half, float);
  else if (d->in_dtype == DAMVS_F16 && od == DAMVS_F16) LAUNCH(__half, __half);
  else return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d direct: in_dtype %d -> out_dtype %d not supported", d->in_dtype, d->out_dtype);
#undef LAUNCH
#undef LAUNCH_V
  DAMVS_LAUNCH_OK("conv3d_direct kernel");
  return DAMVS_OK;
}

size_t conv3d_direct_packed_bytes(const damvs_conv3d_desc* d) {
  return (size_t)((d->Cout + 7) / 8) * 27 * d->Cin * 8 * sizeof(float);
}

int conv3d_direct_pack(const damvs_conv3d_desc* d, const float* weight, void* packed, cudaStream_t st) {
  int total = ((d->Cout + 7) / 8) * 27 * d->Cin * 8;
  pack_weight_direct_kernel<<<(total + 255) / 256, 256, 0, st>>>(weight, (float*)packed, d->Cin, d->Cout,
                                                                 d->transposed, total);
  DAMVS_LAUNCH_OK("pack_weight_direct kernel");
  return DAMVS_OK;
}

}  // namespace damvs
