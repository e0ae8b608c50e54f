// tcgen05 / TMEM implicit-GEMM stride-1 convolution with the depth taps folded into N ("kd-fold").
//
// Same operation and data layout as conv3d_tc.cu (out = skip + relu(conv(in) * scale + shift), G8 bf16 volumes,
// TMA plane loads, kw folded into N and recombined by two shuffles in the epilogue) for the layers with at most 16
// output channels (CostRegNet conv0, conv2, prob and the adjoint convolutions of that shape, reference
// models/module.py:513-530).  Measured on those layers (phase knock-out experiments, DESIGN.md section 3.2): the MMA
// phase alone takes as long as the whole kernel, at ~66 cycles per M128 x N48 x K16 instruction of which ~32 are
// the 4 KB A-operand read from shared memory -- every input plane is read 9 times, once per (kd, kh) tap.
// Here an iteration is one INPUT plane: its three (kh) tap reads feed all three depth taps at once,
//     Y[kd][kw][m] = sum_{kh,ci} in_p[m shifted by kh] * W[kd,kh,kw]          one MMA, N = 3 (kd) x 3 (kw) x 16
// and the result is added into the accumulators of the three output planes z = p + 1 - kd, which live in a ring of
// four 48-column TMEM slots (slot = z mod 4; consecutive planes are consecutive column blocks, so one MMA covers
// them unless the ring wraps, in which case it is issued as two with N = 48 / 96).  A-operand traffic and MMA count
// drop 3x; the B operand (weights) grows to 144 rows, still a few KB.  Slots are zeroed by the epilogue after it
// drains them (tcgen05.st), so every MMA accumulates and no per-slot "first tap" bookkeeping is needed.
//
// Warp roles (320 threads): warp 0 TMA producer, warp 1 MMA issuer, warps 2-9 epilogue: the two warps of a TMEM
// lane quarter alternate output planes, so two planes are drained concurrently while the MMAs of the next two run.
// Barriers: full[slot] (TMA -> MMA), done[slot] (ONE tcgen05.commit per iteration: it frees the plane's slot for the
// producer and tells the epilogue that output plane p - 1 is complete) and acc_empty[ring slot] (epilogue -> MMA).
#include <algorithm>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace damvs {

using namespace tc;

namespace tcf {

constexpr int kP = 32;           // patch pitch in voxels (one TMA box row = 32 voxels * 16 B)
constexpr int RING = 4;          // accumulator slots
constexpr int TMEM_COLS = 256;   // MC * RING * NB <= 256: two CTAs per SM
constexpr int TW = 30;
constexpr int kMaxSlots = 12;
// Two shapes.  Cout <= 8 (conv0, prob): kw blocks of 8 channels, NB = 32 accumulator columns per output plane (24
// used), two 128-row chunks per tile (MC = 2: each epilogue warp drains two units at once, which is what hides its
// TMEM-load / shuffle latencies).  Cout <= 16 (conv2): kw blocks of 16, NB = 48, MC = 1.
template <int CPN> struct Shape {
  static constexpr int NB = CPN == 8 ? 32 : 48;   // columns of one output plane's accumulator (kw folded)
  static constexpr int N3 = 3 * NB;                // full fold: 3 depth taps
  static constexpr int MC = CPN == 8 ? 2 : 1;
  static constexpr int R0 = 4 * MC + 2;            // patch rows: output rows + halo
  static constexpr int TH = 4 * MC;
};
constexpr uint32_t kMagicF = 0x44544346u;  // "DTCF"

struct Header {  // 64 bytes
  uint32_t magic;
  int32_t Cin, Cout, nsteps, pad[12];
};

struct Params {
  const uint8_t* blob;
  const float* scale;
  const float* shift;
  const uint16_t* skip;   // 2-byte elements, same type (bf16 / fp16) as the output volume
  void* out;
  int B, D, H, W;            // stride 1: input extents = output extents
  int Cout, out_G, relu, plain_out, log_nslots, tiles_x, tiles_y, ntiles;
};

__host__ __device__ constexpr int nsteps_of(int G) { return G == 1 ? 2 : 3 * (G / 2); }

__device__ __forceinline__ void tmem_st8_zero(uint32_t taddr) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(taddr), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float shfl_dn(uint32_t v, int d) { return __uint_as_float(__shfl_down_sync(0xffffffffu, v, d)); }

template <int G, int CPN, bool F16>
__global__ void __launch_bounds__(320) conv3d_tcf_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ Params P) {
  using S_ = Shape<CPN>;
  using HT = typename HalfT<F16>::type;
  constexpr int NB = S_::NB, N3 = S_::N3, MC = S_::MC, R0 = S_::R0, TH = S_::TH, CP = CPN;
  constexpr int NSTEPS = nsteps_of(G);
  constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);   // SBO = 128 B, descriptor version 1
  extern __shared__ __align__(1024) uint8_t smem[];
  const int slot_bytes = G * R0 * kP * 16;
  const int nslots = 1 << P.log_nslots;   // 4 or 8
  uint8_t* sA = smem;
  uint8_t* sB = sA + nslots * slot_bytes;                   // [NSTEPS][2][N3][16 B]
  float* sScale = reinterpret_cast<float*>(sB + NSTEPS * 2 * N3 * 16);
  float* sShift = sScale + 16;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sShift + 16);
  uint64_t* full = bars;                      // TMA -> MMA: plane landed
  uint64_t* done = bars + kMaxSlots;          // MMA -> TMA and epilogue: the iteration's MMAs have completed
  uint64_t* acc_empty = bars + 2 * kMaxSlots; // epilogue -> MMA: accumulator slot drained and zeroed
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + RING);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Header* hdr = reinterpret_cast<const Header*>(P.blob);
  if (hdr->magic != kMagicF || hdr->nsteps != NSTEPS || hdr->pad[0] != CPN || hdr->pad[1] != (F16 ? 1 : 0)) {
    if (threadIdx.x == 0 && blockIdx.x == 0) printf("damvs: packed conv weights were not built for the depth-folded kernel\n");
    __trap();
  }
  {
    const uint4* wsrc = reinterpret_cast<const uint4*>(P.blob + sizeof(Header));
    uint4* wdst = reinterpret_cast<uint4*>(sB);
    for (int i = threadIdx.x; i < NSTEPS * 2 * N3; i += blockDim.x) wdst[i] = __ldg(wsrc + i);
    for (int i = threadIdx.x; i < CP; i += blockDim.x) {
      const bool ok = i < P.Cout;
      sScale[i] = ok ? (P.scale ? __ldg(P.scale + i) : 1.f) : 0.f;
      sShift[i] = ok && P.shift ? __ldg(P.shift + i) : 0.f;
    }
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < nslots; ++i) { mbar_init(&full[i], 1); mbar_init(&done[i], 1); }
    for (int i = 0; i < RING; ++i) mbar_init(&acc_empty[i], 4);
    fence_barrier_init();
    tma_prefetch_desc(&map0);
  }
  if (warp == 1) tmem_alloc(tmem_ptr, TMEM_COLS);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // zero the accumulator ring: the two warps of a lane quarter take half of the columns each
  if (warp >= 2) {
    const int q = warp & 3, h = (warp - 2) >> 2;
    constexpr int HALF = MC * RING * NB / 2;
    const uint32_t t0 = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)h * HALF;
#pragma unroll
    for (int c = 0; c < HALF; c += 8) tmem_st8_zero(t0 + c);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const int D = P.D;
#define TILE_COORDS(tile_)                                   \
  const int b = (tile_) / (P.tiles_x * P.tiles_y);           \
  const int ty0 = (((tile_) / P.tiles_x) % P.tiles_y) * TH;  \
  const int tx0 = ((tile_) % P.tiles_x) * TW;

  if (warp == 0) {
    // ===== TMA producer: one input plane per iteration (padding planes are never loaded) =====
    if (lane == 0) {
      int slot = 0, round = 0;
      for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
        TILE_COORDS(tile)
        for (int p = 0; p < D; ++p) {
          if (round > 0) mbar_wait(&done[slot], (round - 1) & 1);
          mbar_arrive_expect_tx(&full[slot], (uint32_t)slot_bytes);
          tma_load_4d(sA + slot * slot_bytes, &map0, &full[slot], (tx0 - 1) * 8, ty0 - 1, p, b * G);
          if (++slot == nslots) { slot = 0; ++round; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const bool leader = elect_one();
    const uint32_t a_base16 = smem_u32(sA) >> 4, b_base16 = smem_u32(sB) >> 4;
    const uint32_t slot16 = (uint32_t)slot_bytes >> 4;
    int slot = 0, round = 0;
    long long zb = 0;   // outputs produced by this CTA before the current tile (ring position of the tile's plane 0)
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x, zb += D) {
      for (int p = 0; p < D; ++p) {
        mbar_wait(&full[slot], round & 1);
        // accumulator slots whose first contribution comes from this plane must have been drained and zeroed
        // (at the end of a tile this is the next tile's plane 0, so a tile's first iteration need not wait again)
        {
          const long long g1 = zb + p + 1;
          if (g1 >= RING) mbar_wait(&acc_empty[g1 & 3], (uint32_t)(((g1 >> 2) - 1) & 1));
        }
        tc_fence_after();
        // blocks j = 0,1,2 <-> kd = 2,1,0 <-> output plane p - 1 + j; B rows are stored in this order
        const int j0 = p == 0 ? 1 : 0, j1 = p == D - 1 ? 2 : 3;
        const int s0 = (int)((zb + p - 1 + j0) & 3);
        const int run1 = min(j1 - j0, RING - s0), run2 = (j1 - j0) - run1;
        const uint32_t so = a_base16 + slot * slot16;
#pragma unroll
        for (int st = 0; st < NSTEPS; ++st) {
          uint32_t a_off16, lbo16;
          if (G == 1) { a_off16 = st == 0 ? 0u : (uint32_t)kP; lbo16 = kP; }                 // (kh0, kh1), (kh1 * 0, kh2)
          else { const int kh = st / (G / 2), gp = st % (G / 2); a_off16 = (uint32_t)((2 * gp * R0 + kh) * kP); lbo16 = R0 * kP; }
          const uint32_t bstep16 = b_base16 + st * (2 * N3);
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int len = r == 0 ? run1 : run2;
            if (len == 0) continue;
            const int jb = r == 0 ? j0 : j0 + run1, sl = r == 0 ? s0 : 0;
            const uint64_t bdesc = ((uint64_t)DESC_HI << 32) | ((bstep16 + jb * NB) | ((uint32_t)N3 << 16));   // LBO = N3 * 16 B
            const uint32_t idesc = len == 3 ? idesc_m128<F16>(N3) : (len == 2 ? idesc_m128<F16>(2 * NB) : idesc_m128<F16>(NB));
#pragma unroll
            for (int c = 0; c < MC; ++c) {
              const uint64_t adesc = ((uint64_t)DESC_HI << 32) | ((so + a_off16 + c * 128) | (lbo16 << 16));
              if (leader) mma_bf16_ss(tmem_base + (c * RING + sl) * NB, adesc, bdesc, idesc, 1u);
            }
          }
        }
        // one commit: the plane can be overwritten (producer), output plane p - 1 -- and D - 1 at the end -- is complete (epilogue)
        if (leader) mma_commit(&done[slot]);
        if (++slot == nslots) { slot = 0; ++round; }
        __syncwarp();
      }
    }
  } else {
    // ===== epilogue: warp (q, h) drains the output planes with global index parity h from TMEM lanes 32q.. =====
    const int q = warp & 3, h = (warp - 2) >> 2;
    constexpr int CPG = CP / 8;
    constexpr int U = MC * CPG;   // (chunk, channel group) units of this warp per output plane
    const int ngroups = P.plain_out ? 1 : min(CPG, (P.Cout + 7) / 8);
    const long long HW = (long long)P.H * P.W;
    const size_t z_stride = (size_t)HW * (P.plain_out ? 1 : 8);
    long long zb = 0;
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x, zb += D) {
      TILE_COORDS(tile)
      bool valid[MC];
      size_t offs[U];
#pragma unroll
      for (int c = 0; c < MC; ++c) {
        const int yo = ty0 + c * 4 + q, xo = tx0 + lane;
        valid[c] = lane < TW && yo < P.H && xo < P.W;
#pragma unroll
        for (int ng = 0; ng < CPG; ++ng)
          offs[c * CPG + ng] = P.plain_out ? (size_t)((long long)b * D * HW + (long long)yo * P.W + xo) : g8_offset(b, ng, 0, yo, xo, P.out_G, D, P.H, P.W);
      }
      for (int z = 0; z < D; ++z) {
        const long long gz = zb + z;
        if ((int)(gz & 1) != h) continue;
        const int sl = (int)(gz & 3);
        const uint32_t tq = tmem_base + ((uint32_t)(32 * q) << 16);
        const uint32_t g = (uint32_t)zb + min(z + 1, D - 1);   // the iteration that completes plane z
        uint4 sk[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          sk[u] = (P.skip && valid[u / CPG] && (u % CPG) < ngroups) ? __ldg(reinterpret_cast<const uint4*>(P.skip + offs[u] + (size_t)z * z_stride)) : make_uint4(0, 0, 0, 0);
        mbar_wait(&done[g & (nslots - 1)], (g >> P.log_nslots) & 1u);
        tc_fence_after();
        if (P.plain_out) {
          uint32_t y0[MC], y1[MC], y2[MC];
#pragma unroll
          for (int c = 0; c < MC; ++c) {
            const uint32_t tbase = tq + (c * RING + sl) * NB;
            tmem_ld1(tbase, y0[c]);
            tmem_ld1(tbase + CP, y1[c]);
            tmem_ld1(tbase + 2 * CP, y2[c]);
          }
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < MC; ++c) {
            const float v = __uint_as_float(y0[c]) + shfl_dn(y1[c], 1) + shfl_dn(y2[c], 2);
            if (valid[c]) reinterpret_cast<float*>(P.out)[offs[c * CPG] + (size_t)z * z_stride] = v;
          }
        } else {
          // all of this warp's TMEM loads are issued before the first use (latency of one, not of U)
          uint32_t y0[U][8], y1[U][8], y2[U][8];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if ((u % CPG) >= ngroups) continue;   // uniform
            const uint32_t tbase = tq + ((u / CPG) * RING + sl) * NB + (u % CPG) * 8;
            tmem_ld8(tbase, y0[u]);
            tmem_ld8(tbase + CP, y1[u]);
            tmem_ld8(tbase + 2 * CP, y2[u]);
          }
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int ng = u % CPG;
            if (ng >= ngroups) continue;   // uniform
            F8 r;
            const uint32_t sw[4] = {sk[u].x, sk[u].y, sk[u].z, sk[u].w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float a = __uint_as_float(y0[u][j]) + shfl_dn(y1[u][j], 1) + shfl_dn(y2[u][j], 2);
              a = a * sScale[ng * 8 + j] + sShift[ng * 8 + j];
              if (P.relu) a = fmaxf(a, 0.f);
              const uint32_t w = sw[j >> 1];
              r.v[j] = a + ((j & 1) ? unpack_hi<F16>(w) : unpack_lo<F16>(w));
            }
            if (valid[u / CPG]) store8(reinterpret_cast<HT*>(P.out) + offs[u] + (size_t)z * z_stride, r);
          }
        }
        // hand the slot back zeroed: the next plane that lands in it accumulates from zero
#pragma unroll
        for (int c = 0; c < MC; ++c)
#pragma unroll
          for (int k = 0; k < NB; k += 8) tmem_st8_zero(tq + (c * RING + sl) * NB + k);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[sl]);
      }
    }
  }
#undef TILE_COORDS
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// B operand of step st: [2 K-halves][N3 rows][8 channels] bf16; row n = j * 48 + kw * 16 + co with j = 2 - kd.
__global__ void pack_weight_tcf_kernel(const float* __restrict__ w, uint8_t* __restrict__ blob, const __grid_constant__ Header hdr, int Cin, int Cout,
                                       int G, int nsteps, int CP, int NB, int f16) {
  const int N3 = 3 * NB;
  uint16_t* dst = reinterpret_cast<uint16_t*>(blob + sizeof(Header));
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // over [nsteps][2][N3][8]
  if (i == 0) *reinterpret_cast<Header*>(blob) = hdr;     // by-value argument: no staging copy, no synchronisation
  if (i >= nsteps * 2 * N3 * 8) return;
  const int j8 = i & 7, n = (i >> 3) % N3, hh = (i / (8 * N3)) & 1, st = i / (16 * N3);
  const int kd = 2 - n / NB, kw = (n % NB) / CP, co = (n % NB) % CP;
  int kh, g;
  bool zero = false;
  if (G == 1) { g = 0; if (st == 0) kh = hh; else { kh = hh + 1; zero = hh == 0; } }
  else { kh = st / (G / 2); g = 2 * (st % (G / 2)) + hh; }
  const int ci = g * 8 + j8;
  float v = 0.f;
  if (!zero && kw < 3 && co < Cout) v = w[((size_t)co * Cin + ci) * 27 + (kd * 3 + kh) * 3 + kw];
  dst[i] = f16 ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

static int cpn_of(const damvs_conv3d_desc* d) { return (d->plain_out || d->Cout <= 8) ? 8 : 16; }
static size_t fixed_smem(int G, int N3) { return (size_t)nsteps_of(G) * 2 * N3 * 16 + 2 * 16 * sizeof(float) + (2 * kMaxSlots + 2 * RING) * sizeof(uint64_t) + 16; }

template <int G, int CPN, bool F16>
static int launch_g(const damvs_conv3d_desc* d, Params& P, const void* in, cudaStream_t st) {
  using S_ = Shape<CPN>;
  constexpr int R0 = S_::R0, TH = S_::TH;
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(DAMVS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  CUtensorMap m0;
  cuuint64_t dims[4] = {(cuuint64_t)d->Win * 8, (cuuint64_t)d->Hin, (cuuint64_t)d->Din, (cuuint64_t)d->B * G};
  cuuint64_t strides[3] = {(cuuint64_t)d->Win * 16, (cuuint64_t)d->Hin * d->Win * 16, (cuuint64_t)d->Din * d->Hin * d->Win * 16};
  cuuint32_t box[4] = {(cuuint32_t)kP * 8, (cuuint32_t)R0, 1, (cuuint32_t)G};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(&m0, F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(in), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(DAMVS_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  const size_t sb = (size_t)G * R0 * kP * 16, fx = fixed_smem(G, S_::N3);
  // ring of 8 planes when two CTAs per SM still fit, else 4 (a power of two: the epilogue maps an iteration to its slot)
  const size_t room = ((227 * 1024) / 2 - fx - 1024) / sb;
  P.log_nslots = room >= 8 ? 3 : 2;
  const int nslots = 1 << P.log_nslots;
  const size_t smem = fx + (size_t)nslots * sb;
  auto kern = conv3d_tcf_kernel<G, CPN, F16>;
  DAMVS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DAMVS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  P.tiles_x = (d->Win + TW - 1) / TW;
  P.tiles_y = (d->Hin + TH - 1) / TH;
  P.ntiles = P.tiles_x * P.tiles_y * d->B;
  dim3 grid((unsigned)std::min(P.ntiles, 2 * current_sm_count()), 1, 1);   // two CTAs per SM (256 TMEM columns each)
  kern<<<grid, 320, smem, st>>>(m0, P);
  DAMVS_LAUNCH_OK("conv3d_tcf kernel");
  return DAMVS_OK;
}

}  // namespace tcf

// ---- entry points used by conv3d_tc.cu's dispatch ------------------------------------------------------------------
bool conv3d_tcf_supported(const damvs_conv3d_desc* d) {
  if (d->transposed || d->stride != 1 || d->Cout > 16 || d->Cin % 8) return false;
  const int G = d->Cin / 8;
  return G == 1 || G == 2 || G == 4;
}

size_t conv3d_tcf_packed_bytes(const damvs_conv3d_desc* d) {
  const int n3 = tcf::cpn_of(d) == 8 ? tcf::Shape<8>::N3 : tcf::Shape<16>::N3;
  return (sizeof(tcf::Header) + (size_t)tcf::nsteps_of(d->Cin / 8) * 2 * n3 * 16 + 255) / 256 * 256;
}

int conv3d_tcf_pack(const damvs_conv3d_desc* d, const float* weight, void* packed, cudaStream_t st) {
  const int G = d->Cin / 8, nsteps = tcf::nsteps_of(G);
  tcf::Header h{};
  const int cpn = tcf::cpn_of(d), nb = cpn == 8 ? tcf::Shape<8>::NB : tcf::Shape<16>::NB;
  h.magic = tcf::kMagicF; h.Cin = d->Cin; h.Cout = d->Cout; h.nsteps = nsteps; h.pad[0] = cpn; h.pad[1] = d->in_dtype == DAMVS_F16 ? 1 : 0;
  const int total = nsteps * 2 * 3 * nb * 8;
  tcf::pack_weight_tcf_kernel<<<(total + 255) / 256, 256, 0, st>>>(weight, (uint8_t*)packed, h, d->Cin, d->plain_out ? 1 : d->Cout, G, nsteps, cpn, nb,
                                                                   d->in_dtype == DAMVS_F16 ? 1 : 0);
  DAMVS_LAUNCH_OK("pack_weight_tcf kernel");
  return DAMVS_OK;
}

int conv3d_tcf_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, const float* scale, const float* shift,
                      const void* skip, void* out, cudaStream_t st) {
  tcf::Params P{};
  P.blob = (const uint8_t*)packed; P.scale = scale; P.shift = shift; P.skip = (const uint16_t*)skip; P.out = out;
  P.B = d->B; P.D = d->Din; P.H = d->Hin; P.W = d->Win;
  P.Cout = d->plain_out ? 1 : d->Cout; P.out_G = d->plain_out ? 1 : (d->Cout + 7) / 8; P.relu = d->relu; P.plain_out = d->plain_out;
  const int G = d->Cin / 8;
  const bool f16 = d->in_dtype == DAMVS_F16;
#define GO(G_, CPN_) return f16 ? tcf::launch_g<G_, CPN_, true>(d, P, in, st) : tcf::launch_g<G_, CPN_, false>(d, P, in, st)
  if (tcf::cpn_of(d) == 8) {
    if (G == 1) GO(1, 8);
    if (G == 2) GO(2, 8);
    if (G == 4) GO(4, 8);
  } else {
    if (G == 1) GO(1, 16);
    if (G == 2) GO(2, 16);
    if (G == 4) GO(4, 16);
  }
#undef GO
  return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05 (depth-folded): Cin=%d not supported", d->Cin);
}

}  // namespace damvs
