// tcgen05 / TMEM implicit-GEMM 3x3x3 convolution blocks of CostRegNet (bf16 in, fp32 accumulate).
//
// Replaces Conv3d / Deconv3d (reference models/module.py:117-202: nn.Conv3d /
// nn.ConvTranspose3d + BatchNorm3d + ReLU) and the skip-adds of CostRegNet.forward
// (models/module.py:532-541) with one kernel per layer:
//     out = skip + relu(conv(in) * scale + shift)
//
// GEMM view.  M = voxels of a (4*MC rows x 32 columns) tile of one depth plane, K = 9 * Cin (the
// (kd, kh) taps), N = 3 * CP: the three kw taps are folded into the N dimension (CP = Cout padded to
// 16/32/64), i.e. the MMA computes Y_kw[m] = sum_{kd,kh,ci} in[m shifted by (kd,kh)] * W[kd,kh,kw]
// for kw = 0..2 at once and the epilogue adds out[x] = Y_0[x] + Y_1[x+1] + Y_2[x+2] with two warp
// shuffles (a tile row is 32 GEMM rows = one warp's TMEM lanes, of which 30 are real outputs).
// Why: with both operands in shared memory a K=16 MMA re-reads its 128x16 A tile (4 KB, 32 cycles of
// shared-memory bandwidth) whatever N is, so at N = Cout = 8..16 the un-folded form is bound by A
// reads, not by the tensor pipe; folding kw cuts the A reads (and MMA count) by 3.
//
// The A operand is never materialised (no im2col):
//   * activations live in the G8 layout ([B][C/8][D][H][W][8] bf16), so an 8-channel group of a
//     (rows x 32 voxels) patch of one depth plane lands in shared memory, via ONE TMA box load with
//     a contiguous 512-byte inner dimension, as a dense array of 16-byte rows -- exactly the
//     no-swizzle K-major UMMA layout (8-row x 16-byte core matrices, SBO = 128 B);
//   * GEMM row m = ty*32 + tx; a (kh) tap is the SAME shared-memory patch shifted by kh*32 rows, i.e.
//     a different descriptor start address; the two 8-channel K-halves of one MMA are two such
//     addresses LBO bytes apart (the next channel group's plane, or -- for Cin = 8 -- the next tap);
//   * depth taps come from a ring of plane slots that slides along D, so every input plane is
//     loaded once per CTA; out-of-range planes / rows / columns are TMA zero fill (= padding 1).
//
// Three modes share the kernel: stride-1 conv, stride-2 conv (even/odd input rows as two patches;
// odd output columns computed and dropped) and the k3/s2/p1/op1 transposed conv (4 (d,h)-parity
// classes x the w-parity pair folded into N, each class a 1/2/4-tap sub-convolution of the same
// input patch with its own TMEM accumulator).
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2-9 =
// epilogue (TMEM -> registers -> kw combine -> BN affine / ReLU / skip -> 16-byte stores).
// Accumulators are double buffered in TMEM so the epilogue of plane z overlaps the MMAs of plane z+1.
#include <algorithm>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace damvs {

using namespace tc;

constexpr int kP = 32;         // patch pitch in voxels (one TMA box row = 32 voxels * 16 B)
constexpr int kMaxSlots = 16;  // depth-plane ring (actual depth chosen per launch)
// Accumulator buffers in TMEM: two when they fit -- except the 16-channel transposed layers (conv9, conv11: 192 columns),
// which run single-buffered in 256 columns so that two CTAs share an SM instead of one double-buffered CTA in 512: their
// epilogue (8 output positions per input voxel) is the long phase, and 16 epilogue warps per SM hide its latencies better
// than 8 (conv11 128/124/57 -> 105/108/50 us at stages 3/2/1; no change with four views in flight).
__host__ __device__ constexpr int nbuf_of(int mode, int cp, int acc_cols) {
  return (mode == 2 && cp == 16 && acc_cols == 192) ? 1 : (2 * acc_cols <= 512 ? 2 : 1);
}
constexpr int kMaxSteps = 96;
constexpr uint32_t kMagic = 0x44544332u;  // "DTC2"

enum { MODE_S1 = 0, MODE_S2 = 1, MODE_T = 2 };

// One K=16 MMA of the per-iteration program, in layer-independent form (host-built, stored in the packed buffer).
struct StepSrc {
  int8_t slot_rel, cls, first, pad_;
  int8_t patch[2], g[2], dy[2], tap[2];  // per K-half; tap = kd*3+kh (td*3+th for transposed), < 0 => zero weights
};
struct PackedHeader {  // 64 bytes
  uint32_t magic;
  int32_t mode, Cin, Cout, CP, nsteps, ncls, n0;  // n0: first output channel this blob computes
  int32_t blob_bytes, nblobs, f16, pad[5];   // f16: weights are IEEE half (1) or bfloat16 (0)
};

struct TcParams {
  const uint8_t* blob;  // PackedHeader + StepSrc[nsteps] (padded to 16 B) + weights
  const float* scale;
  const float* shift;
  const uint16_t* skip;  // 2-byte elements, same type (bf16 / fp16) as the output volume
  void* out;
  int B, G, Din, Hin, Win, Dout, Hout, Wout;
  int out_G, out_g0;  // output volume's group count and first group written by this launch
  int n0, Cout, relu, plain_out, niter, nsteps, nslots;
  int tiles_x, tiles_y, ntiles;  // persistent CTAs walk tiles blockIdx.x, blockIdx.x + gridDim.x, ...
  int zchunks, zlen;             // a tile covers zlen iterations (depth planes) of one of zchunks depth ranges
};

__host__ __device__ inline int steps_offset() { return (int)sizeof(PackedHeader); }
__host__ __device__ inline int weights_offset(int nsteps) { return (int)sizeof(PackedHeader) + ((nsteps * (int)sizeof(StepSrc) + 15) & ~15); }

template <int MODE>
struct Geo {
  static constexpr int span = MODE == MODE_T ? 2 : 3;
  static constexpr int adv = MODE == MODE_S2 ? 2 : 1;
  static constexpr int p0 = MODE == MODE_T ? 0 : -1;
  static constexpr int ncls = MODE == MODE_T ? 4 : 1;
  static constexpr int TW = MODE == MODE_S1 ? 30 : (MODE == MODE_T ? 31 : 15);
  __host__ __device__ static constexpr int rows0(int MC) { return MODE == MODE_S1 ? 4 * MC + 2 : (MODE == MODE_T ? 4 * MC + 1 : 4 * MC); }
  __host__ __device__ static constexpr int rows1(int MC) { return MODE == MODE_S2 ? 4 * MC + 1 : 0; }
};

__device__ __forceinline__ float shfl_dn(uint32_t v, int d) { return __uint_as_float(__shfl_down_sync(0xffffffffu, v, d)); }


// ---------------------------------------------------------------------------------------------
// The per-iteration MMA program as straight-line code: every operand offset is a compile-time
// constant (MODE, G = Cin/8 and MC are template parameters), only the three plane-slot bases are
// run-time (uniform) values.  The order of the steps is the order build_program() emits on the host,
// which is also the order of the packed B operands.
// ---------------------------------------------------------------------------------------------
template <int N, int MC, bool F16>
__device__ __forceinline__ void issue_step(bool leader, uint32_t so, uint32_t a_off16, uint32_t lbo16, uint32_t b_base16, int step,
                                           uint32_t dcol, uint32_t acc) {
  constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);  // SBO = 128 B, descriptor version 1
  constexpr uint32_t IDESC = idesc_m128<F16>(N);
  const uint64_t bdesc = ((uint64_t)DESC_HI << 32) | ((b_base16 + step * (2 * N)) | ((uint32_t)N << 16));  // LBO = N*16 bytes
#pragma unroll
  for (int c = 0; c < MC; ++c) {
    const uint64_t adesc = ((uint64_t)DESC_HI << 32) | ((so + a_off16 + c * 128) | (lbo16 << 16));
    if (leader) mma_bf16_ss(dcol + c * N, adesc, bdesc, IDESC, acc);
  }
}

template <int MODE, int CP, int MC, int G, bool F16>
__device__ __forceinline__ void issue_iteration(bool leader, uint32_t so0, uint32_t so1, uint32_t so2, uint32_t b_base16, uint32_t dbase) {
  using G_ = Geo<MODE>;
  constexpr int N = 3 * CP;
  constexpr int R0 = G_::rows0(MC), R1 = G_::rows1(MC);
  constexpr uint32_t P0_16 = (uint32_t)G * R0 * kP;  // patch-0 size in 16-byte units
  int step = 0;
  if (MODE == MODE_S1) {
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
      const uint32_t so = kd == 0 ? so0 : (kd == 1 ? so1 : so2);
      if (G == 1) {  // (kh0, kh1), (kh1 with zero weights, kh2)
        issue_step<N, MC, F16>(leader, so, 0, kP, b_base16, step++, dbase, kd == 0 ? 0u : 1u);
        issue_step<N, MC, F16>(leader, so, kP, kP, b_base16, step++, dbase, 1u);
      } else {
#pragma unroll
        for (int kh = 0; kh < 3; ++kh)
#pragma unroll
          for (int gp = 0; gp < G / 2; ++gp)
            issue_step<N, MC, F16>(leader, so, (uint32_t)((2 * gp * R0 + kh) * kP), (uint32_t)(R0 * kP), b_base16, step++, dbase,
                              (kd == 0 && kh == 0 && gp == 0) ? 0u : 1u);
      }
    }
  } else if (MODE == MODE_S2) {
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
      const uint32_t so = kd == 0 ? so0 : (kd == 1 ? so1 : so2);
      if (G == 1) {  // (E row, O row r), (O row r with zero weights, O row r+1)
        issue_step<N, MC, F16>(leader, so, 0, P0_16, b_base16, step++, dbase, kd == 0 ? 0u : 1u);
        issue_step<N, MC, F16>(leader, so, P0_16, kP, b_base16, step++, dbase, 1u);
      } else {
#pragma unroll
        for (int t = 0; t < 3; ++t)  // E (kh=1), O row r (kh=0), O row r+1 (kh=2)
#pragma unroll
          for (int gp = 0; gp < G / 2; ++gp) {
            const uint32_t off = t == 0 ? (uint32_t)(2 * gp * R0 * kP) : P0_16 + (uint32_t)((2 * gp * R1 + (t - 1)) * kP);
            issue_step<N, MC, F16>(leader, so, off, (uint32_t)((t == 0 ? R0 : R1) * kP), b_base16, step++, dbase,
                              (kd == 0 && t == 0 && gp == 0) ? 0u : 1u);
          }
      }
    }
  } else {
    // parity 0 <- one tap (shift 0); parity 1 <- two taps (shift 0, then shift 1)
#pragma unroll
    for (int pd = 0; pd < 2; ++pd)
#pragma unroll
      for (int ph = 0; ph < 2; ++ph) {
        const uint32_t dcol = dbase + (pd * 2 + ph) * MC * N;
        bool first = true;
#pragma unroll
        for (int a = 0; a <= pd; ++a) {        // d taps: shift a
          const uint32_t so = a == 0 ? so0 : so1;
#pragma unroll
          for (int bq = 0; bq <= ph; ++bq)     // h taps: shift bq
#pragma unroll
            for (int gp = 0; gp < G / 2; ++gp) {
              issue_step<N, MC, F16>(leader, so, (uint32_t)((2 * gp * R0 + bq) * kP), (uint32_t)(R0 * kP), b_base16, step++, dcol, first ? 0u : 1u);
              first = false;
            }
        }
      }
  }
}

template <int MODE, int CP, int MC, int G, bool F16>
__global__ void __launch_bounds__(320) conv3d_tc_kernel(const __grid_constant__ CUtensorMap map0,
                                                        const __grid_constant__ CUtensorMap map1,
                                                        const __grid_constant__ TcParams P) {
  using G_ = Geo<MODE>;
  constexpr int N = 3 * CP;
  constexpr int TH = 4 * MC;
  constexpr int ACC_COLS = G_::ncls * MC * N;
  constexpr int NBUF = nbuf_of(MODE, CP, ACC_COLS);
  constexpr int NEED = NBUF * ACC_COLS;
  constexpr int TMEM_COLS = NEED <= 32 ? 32 : NEED <= 64 ? 64 : NEED <= 128 ? 128 : NEED <= 256 ? 256 : 512;
  static_assert(ACC_COLS <= 512, "TMEM budget");
  using HT = typename HalfT<F16>::type;   // element type of the input / output / skip volumes and of the packed weights

  extern __shared__ __align__(1024) uint8_t smem[];
  const int patch0_bytes = G * G_::rows0(MC) * kP * 16;
  const int patch1_bytes = G * G_::rows1(MC) * kP * 16;
  const int slot_stride = patch0_bytes + patch1_bytes;
  const int nslots = P.nslots;
  const PackedHeader* hdr = reinterpret_cast<const PackedHeader*>(P.blob);
  const int nsteps = P.nsteps;
  if (hdr->magic != kMagic || hdr->mode != MODE || hdr->CP != CP || hdr->nsteps != nsteps || hdr->f16 != (F16 ? 1 : 0)) {
    if (threadIdx.x == 0 && blockIdx.x == 0)
      printf("damvs: packed conv weights were built for another layer type (mode %d CP %d, kernel mode %d CP %d)\n", hdr->mode, hdr->CP, MODE, CP);
    __trap();
  }
  uint8_t* sA = smem;
  uint8_t* sB = sA + nslots * slot_stride;
  float* sScale = reinterpret_cast<float*>(sB + nsteps * 2 * N * 16);
  float* sShift = sScale + CP;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sShift + CP);
  uint64_t* full = bars;
  uint64_t* empty = bars + kMaxSlots;
  uint64_t* tmem_full = bars + 2 * kMaxSlots;
  uint64_t* tmem_empty = bars + 2 * kMaxSlots + 2;
  uint64_t* wbar = bars + 2 * kMaxSlots + 4;   // the layer's weights have landed in shared memory
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kMaxSlots + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tile -> (batch item, tile origin); origins are output coords for S1/S2, input coords for T
#define TILE_COORDS(tile_)                                               \
  const int t2_ = (tile_) / P.zchunks;                                   \
  const int it0 = ((tile_) - t2_ * P.zchunks) * P.zlen;                  \
  const int nit = min(P.zlen, P.niter - it0);                            \
  const int b = t2_ / (P.tiles_x * P.tiles_y);                           \
  const int ty0 = ((t2_ / P.tiles_x) % P.tiles_y) * TH;                  \
  const int tx0 = (t2_ % P.tiles_x) * G_::TW;

  // ---- one-time setup ------------------------------------------------------------------------
  // The weights (up to 110 KB for the 64-channel layers) arrive by bulk copies issued below, off the critical path: the
  // per-CTA timelines of the coarse layers showed 4.5-7 us of a 10-15 us CTA life spent in a ld.global / st.shared loop.
  {
    for (int i = threadIdx.x; i < CP; i += blockDim.x) {
      int co = P.n0 + i;
      bool ok = co < P.Cout;
      sScale[i] = ok ? (P.scale ? __ldg(P.scale + co) : 1.f) : 0.f;
      sShift[i] = ok && P.shift ? __ldg(P.shift + co) : 0.f;
    }
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < nslots; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(&tmem_full[0], 1); mbar_init(&tmem_full[1], 1);
    mbar_init(&tmem_empty[0], 8); mbar_init(&tmem_empty[1], 8);
    mbar_init(wbar, 1);
    fence_barrier_init();
    {
      const uint8_t* wsrc = P.blob + weights_offset(nsteps);
      const uint32_t wbytes = (uint32_t)nsteps * 2 * N * 16;
      mbar_arrive_expect_tx(wbar, wbytes);
      for (uint32_t off = 0; off < wbytes; off += 32768) bulk_load(sB + off, wsrc + off, min(32768u, wbytes - off), wbar);
    }
    tma_prefetch_desc(&map0);
    if (MODE == MODE_S2) tma_prefetch_desc(&map1);
  }
  if (warp == 1) tmem_alloc(tmem_ptr, TMEM_COLS);
  fence_proxy_async();  // generic-proxy smem writes (weights) -> visible to the async proxy (UMMA)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int niter = P.niter;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)(patch0_bytes + patch1_bytes);
      int slot = 0, round = 0;
      for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
      TILE_COORDS(tile)
      const int nplanes = (nit - 1) * G_::adv + G_::span;
      for (int k = 0; k < nplanes; ++k) {
        if (round > 0) mbar_wait(&empty[slot], (round - 1) & 1);
        mbar_arrive_expect_tx(&full[slot], bytes);
        uint8_t* dst = sA + slot * slot_stride;
        const int plane = it0 * G_::adv + k + G_::p0;
        if (MODE == MODE_S1) {
          tma_load_4d(dst, &map0, &full[slot], (tx0 - 1) * 8, ty0 - 1, plane, b * G);
        } else if (MODE == MODE_T) {
          tma_load_4d(dst, &map0, &full[slot], tx0 * 8, ty0, plane, b * G);
        } else {
          tma_load_4d(dst, &map0, &full[slot], (2 * tx0 - 1) * 8, ty0, plane, b * G);                    // even rows 2*(ty0+r)
          tma_load_4d(dst + patch0_bytes, &map1, &full[slot], (2 * tx0 - 1) * 8, ty0 - 1, plane, b * G);  // odd rows 2*(ty0+r)-1
        }
        if (++slot == nslots) { slot = 0; ++round; }
      }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp walks the (uniform) program, one elected lane issues =====
    const bool leader = elect_one();
    const uint32_t a_base16 = smem_u32(sA) >> 4, b_base16 = smem_u32(sB) >> 4;
    const uint32_t slot16 = (uint32_t)slot_stride >> 4;
    mbar_wait(wbar, 0);                                      // B operand in place
    int wait_slot = 0, wait_round = 0;                       // full-barrier cursor (runs across tiles)
    int base_slot = 0;                                       // slot of the first plane of this iteration
    int acc_n = 0;                                           // accumulator buffers handed to the epilogue so far
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
    int next_wait = 0;
    const int nit = min(P.zlen, P.niter - (tile % P.zchunks) * P.zlen);
    for (int it = 0; it < nit; ++it, ++acc_n) {
      const int need = it * G_::adv + G_::span - 1;
      while (next_wait <= need) {
        mbar_wait(&full[wait_slot], wait_round & 1);
        ++next_wait;
        if (++wait_slot == nslots) { wait_slot = 0; ++wait_round; }
      }
      const int buf = NBUF == 2 ? (acc_n & 1) : 0;
      if (acc_n >= NBUF) mbar_wait(&tmem_empty[buf], (NBUF == 2 ? ((acc_n >> 1) - 1) : (acc_n - 1)) & 1);
      tc_fence_after();
      const uint32_t dbase = tmem_base + buf * ACC_COLS;
      int s1 = base_slot + 1; if (s1 >= nslots) s1 -= nslots;
      int s2 = base_slot + 2; if (s2 >= nslots) s2 -= nslots;
      const uint32_t so0 = a_base16 + base_slot * slot16;
      const uint32_t so1 = a_base16 + s1 * slot16;
      const uint32_t so2 = a_base16 + s2 * slot16;
      issue_iteration<MODE, CP, MC, G, F16>(leader, so0, so1, so2, b_base16, dbase);
      if (leader) {
        mma_commit(&tmem_full[buf]);
#pragma unroll
        for (int a = 0; a < G_::adv; ++a) {
          int rs = base_slot + a; if (rs >= nslots) rs -= nslots;
          mma_commit(&empty[rs]);
        }
      }
      base_slot += G_::adv; if (base_slot >= nslots) base_slot -= nslots;
      __syncwarp();
    }
    // the last span - adv planes of the tile were only read, never released, by the iteration loop
    if (leader) {
#pragma unroll
      for (int a = 0; a < G_::span - G_::adv; ++a) {
        int rs = base_slot + a; if (rs >= nslots) rs -= nslots;
        mma_commit(&empty[rs]);
      }
    }
    base_slot += G_::span - G_::adv; if (base_slot >= nslots) base_slot -= nslots;
    __syncwarp();
    }
  } else {
    // ===== epilogue: 8 warps; warp w owns TMEM lanes 32*(w%4).., the two warps of a lane quarter split the
    // work units (chunks, or channel groups, or parity classes) of an iteration between them =====
    const int q = warp & 3, half = (warp - 2) >> 2;
    constexpr int CPG = CP / 8;
    const int ngroups = P.plain_out ? 1 : min(CPG, (P.Cout - P.n0 + 7) / 8);   // real (non-padding) channel groups
    const long long HWo = (long long)P.Hout * P.Wout;
    // element stride of one iteration in the output volume (transposed: two output planes per input plane)
    const size_t it_stride = (size_t)HWo * (P.plain_out ? 1 : 8) * (MODE == MODE_T ? 2 : 1);
    constexpr int UT = MODE == MODE_T ? 2 * MC * CPG : 1;
    constexpr int US = MODE == MODE_T ? 1 : (MC >= 2 ? (MC / 2) * CPG : (CPG + 1) / 2);
    int acc_n = 0;
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
    TILE_COORDS(tile)
    // per-tile addressing, hoisted out of the plane loop: offsets of this thread's work units at iteration 0
    // (they advance by it_stride per iteration) and their validity
    size_t offsT[UT], offsS[US];
    bool validT[MC], validS[US];
    if (MODE == MODE_T) {
#pragma unroll
      for (int c = 0; c < MC; ++c) {
        const int yi = ty0 + c * 4 + q, xi = tx0 + lane;
        validT[c] = lane < G_::TW && yi < P.Hin && xi < P.Win;
      }
#pragma unroll
      for (int u = 0; u < UT; ++u) {
        const int k = u / (MC * CPG), c = (u / CPG) % MC, ng = u % CPG;
        const int pdh = 2 * half + k, pd = pdh >> 1, ph = pdh & 1;
        const int yi = ty0 + c * 4 + q, xi = tx0 + lane;
        offsT[u] = g8_offset(b, P.out_g0 + ng, pd, 2 * yi + ph, 2 * xi, P.out_G, P.Dout, P.Hout, P.Wout);
      }
    } else {
#pragma unroll
      for (int u = 0; u < US; ++u) {
        const int c = MC >= 2 ? half * (MC / 2) + u / CPG : 0;
        const int ng = MC >= 2 ? u % CPG : 2 * u + half;
        const int ty = c * 4 + q, tx = lane;
        int yo = ty0 + ty, xo;
        if (MODE == MODE_S1) { xo = tx0 + tx; validS[u] = tx < G_::TW && yo < P.Hout && xo < P.Wout; }
        else { xo = tx0 + (tx >> 1); validS[u] = !(tx & 1) && (tx >> 1) < G_::TW && yo < P.Hout && xo < P.Wout; }
        if (P.plain_out) offsS[u] = (size_t)((long long)b * P.Dout * HWo + (long long)yo * P.Wout + xo);
        else offsS[u] = g8_offset(b, P.out_g0 + ng, 0, yo, xo, P.out_G, P.Dout, P.Hout, P.Wout);
      }
    }
#pragma unroll
    for (int u = 0; u < UT; ++u) offsT[u] += (size_t)it0 * it_stride;
#pragma unroll
    for (int u = 0; u < US; ++u) offsS[u] += (size_t)it0 * it_stride;
    for (int it = 0; it < nit; ++it, ++acc_n) {
      const int buf = NBUF == 2 ? (acc_n & 1) : 0;
      const uint32_t tbase = tmem_base + ((uint32_t)(32 * q) << 16) + buf * ACC_COLS;
      if (MODE == MODE_T) {
        // units: (class pdh in {2*half, 2*half+1}) x chunk x group; each unit = two adjacent output voxels (x parity)
        constexpr int U = 2 * MC * CPG;
        uint4 sk[U][2];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int c = (u / CPG) % MC, ng = u % CPG;
          if (P.skip && validT[c] && ng < ngroups) {
            sk[u][0] = __ldg(reinterpret_cast<const uint4*>(P.skip + offsT[u]));
            sk[u][1] = __ldg(reinterpret_cast<const uint4*>(P.skip + offsT[u] + 8));
            // the same voxels two output planes further are next iteration's skip operands: start them towards L1
            // now, a whole iteration ahead (this wait is short when the epilogue is the slower stage)
            if (it + 1 < nit)
              asm volatile("prefetch.global.L1 [%0];" ::"l"(P.skip + offsT[u] + it_stride));
          } else {
            sk[u][0] = sk[u][1] = make_uint4(0, 0, 0, 0);
          }
        }
        mbar_wait(&tmem_full[buf], (NBUF == 2 ? (acc_n >> 1) : acc_n) & 1);
        tc_fence_after();
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int k = u / (MC * CPG), c = (u / CPG) % MC, ng = u % CPG;
          if (ng >= ngroups) continue;   // uniform
          const int pdh = 2 * half + k;
          const uint32_t cbase = tbase + (pdh * MC + c) * N + ng * 8;
          uint32_t ya[8], yb[8], yc[8];  // tw = 1 (even x), tw = 2 (odd x, same input), tw = 0 (odd x, input + 1)
          tmem_ld8(cbase, ya);
          tmem_ld8(cbase + CP, yb);
          tmem_ld8(cbase + 2 * CP, yc);
          tmem_ld_wait();
          F8 r0, r1;
          const uint32_t s0[4] = {sk[u][0].x, sk[u][0].y, sk[u][0].z, sk[u][0].w};
          const uint32_t s1[4] = {sk[u][1].x, sk[u][1].y, sk[u][1].z, sk[u][1].w};
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float a = __uint_as_float(ya[j]);
            float bb = __uint_as_float(yb[j]) + shfl_dn(yc[j], 1);
            a = a * sScale[ng * 8 + j] + sShift[ng * 8 + j];
            bb = bb * sScale[ng * 8 + j] + sShift[ng * 8 + j];
            if (P.relu) { a = fmaxf(a, 0.f); bb = fmaxf(bb, 0.f); }
            const uint32_t w0 = s0[j >> 1], w1 = s1[j >> 1];
            r0.v[j] = a + ((j & 1) ? unpack_hi<F16>(w0) : unpack_lo<F16>(w0));
            r1.v[j] = bb + ((j & 1) ? unpack_hi<F16>(w1) : unpack_lo<F16>(w1));
          }
          if (validT[c]) {
            HT* o = reinterpret_cast<HT*>(P.out) + offsT[u];
            store8(o, r0);
            store8(o + 8, r1);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) offsT[u] += it_stride;
      } else {
        constexpr int U = US;
        uint4 sk[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int ng = MC >= 2 ? u % CPG : 2 * u + half;
          sk[u] = (P.skip && validS[u] && ng < ngroups) ? __ldg(reinterpret_cast<const uint4*>(P.skip + offsS[u])) : make_uint4(0, 0, 0, 0);
        }
        mbar_wait(&tmem_full[buf], (NBUF == 2 ? (acc_n >> 1) : acc_n) & 1);
        tc_fence_after();
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int c = MC >= 2 ? half * (MC / 2) + u / CPG : 0;
          const int ng = MC >= 2 ? u % CPG : 2 * u + half;
          if (ng >= ngroups) continue;   // uniform
          const uint32_t cbase = tbase + c * N + ng * 8;
          if (P.plain_out) {
            uint32_t y0, y1, y2;
            tmem_ld1(cbase, y0);
            tmem_ld1(cbase + CP, y1);
            tmem_ld1(cbase + 2 * CP, y2);
            tmem_ld_wait();
            const float v = __uint_as_float(y0) + shfl_dn(y1, 1) + shfl_dn(y2, 2);
            if (validS[u]) reinterpret_cast<float*>(P.out)[offsS[u]] = v;
          } else {
            uint32_t y0[8], y1[8], y2[8];
            tmem_ld8(cbase, y0);
            tmem_ld8(cbase + CP, y1);
            tmem_ld8(cbase + 2 * CP, y2);
            tmem_ld_wait();
            F8 r;
            const uint32_t sw[4] = {sk[u].x, sk[u].y, sk[u].z, sk[u].w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float a = __uint_as_float(y0[j]) + shfl_dn(y1[j], 1) + shfl_dn(y2[j], 2);
              a = a * sScale[ng * 8 + j] + sShift[ng * 8 + j];
              if (P.relu) a = fmaxf(a, 0.f);
              const uint32_t w = sw[j >> 1];
              r.v[j] = a + ((j & 1) ? unpack_hi<F16>(w) : unpack_lo<F16>(w));
            }
            if (validS[u]) store8(reinterpret_cast<HT*>(P.out) + offsS[u], r);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) offsS[u] += it_stride;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
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

// ---------------------------------------------------------------------------------------------
// host side: per-layer MMA program, weight packing, tensor maps, launch
// ---------------------------------------------------------------------------------------------
static int mode_of(const damvs_conv3d_desc* d) { return d->transposed ? MODE_T : (d->stride == 2 ? MODE_S2 : MODE_S1); }
static int padded_c(int cout) { return cout <= 16 ? 16 : (cout <= 32 ? 32 : 64); }

struct Half { int patch, g, dy, tap; };

static bool build_program(int mode, int G, std::vector<StepSrc>& steps) {
  steps.clear();
  if (G != 1 && G % 2 != 0) return false;
  auto emit = [&](int slot_rel, int cls, bool first, const Half& a, const Half& b2) {
    StepSrc s{};
    s.slot_rel = (int8_t)slot_rel; s.cls = (int8_t)cls; s.first = first ? 1 : 0;
    const Half* h[2] = {&a, &b2};
    for (int i = 0; i < 2; ++i) {
      s.patch[i] = (int8_t)h[i]->patch; s.g[i] = (int8_t)h[i]->g; s.dy[i] = (int8_t)h[i]->dy; s.tap[i] = (int8_t)h[i]->tap;
    }
    steps.push_back(s);
  };
  // `taps` of one (class, slot) group must be listed in increasing shared-memory offset so that LBO > 0
  auto emit_group = [&](int slot_rel, int cls, bool& first, std::vector<Half>& taps) {
    if (G % 2 == 0) {
      for (const Half& t : taps)
        for (int g = 0; g < G; g += 2) {
          Half a = t, b2 = t;
          a.g = g; b2.g = g + 1;
          emit(slot_rel, cls, first, a, b2);
          first = false;
        }
    } else {  // G == 1 (Cin = 8): a K=16 MMA spans two taps; an odd tail re-reads the previous tap with zero weights
      for (size_t i = 0; i < taps.size(); i += 2) {
        Half a, b2;
        if (i + 1 < taps.size()) { a = taps[i]; b2 = taps[i + 1]; }
        else if (i > 0) { a = taps[i - 1]; a.tap = -1; b2 = taps[i]; }
        else return false;
        emit(slot_rel, cls, first, a, b2);
        first = false;
      }
    }
    return true;
  };
  bool ok = true;
  if (mode == MODE_S1) {
    bool first = true;
    for (int kd = 0; kd < 3; ++kd) {
      std::vector<Half> taps;
      for (int kh = 0; kh < 3; ++kh) taps.push_back({0, 0, kh, kd * 3 + kh});
      ok = ok && emit_group(kd, 0, first, taps);
    }
  } else if (mode == MODE_S2) {
    bool first = true;
    for (int kd = 0; kd < 3; ++kd) {
      std::vector<Half> taps;  // even-row patch (kh = 1) first, then the odd-row patch (kh = 0 at row r, kh = 2 at row r+1)
      taps.push_back({0, 0, 0, kd * 3 + 1});
      taps.push_back({1, 0, 0, kd * 3 + 0});
      taps.push_back({1, 0, 1, kd * 3 + 2});
      ok = ok && emit_group(kd, 0, first, taps);
    }
  } else {
    if (G % 2) return false;
    // output o = 2*i - 1 + t: parity 0 <- (t=1, i=j); parity 1 <- (t=2, i=j), (t=0, i=j+1)
    auto dim_taps = [](int p, int (&t)[2], int (&s)[2]) { if (p == 0) { t[0] = 1; s[0] = 0; return 1; } t[0] = 2; s[0] = 0; t[1] = 0; s[1] = 1; return 2; };
    for (int pd = 0; pd < 2; ++pd)
      for (int ph = 0; ph < 2; ++ph) {
        const int cls = pd * 2 + ph;
        bool first = true;
        int td[2], sd[2], th[2], sh[2];
        int nd = dim_taps(pd, td, sd), nh = dim_taps(ph, th, sh);
        for (int a = 0; a < nd; ++a) {
          std::vector<Half> taps;
          for (int bq = 0; bq < nh; ++bq) taps.push_back({0, 0, sh[bq], td[a] * 3 + th[bq]});
          ok = ok && emit_group(sd[a], cls, first, taps);
        }
      }
  }
  return ok && (int)steps.size() <= kMaxSteps;
}

// depth-folded variant for stride-1 layers with <= 16 output channels (conv3d_tcf.cu)
bool conv3d_tcf_supported(const damvs_conv3d_desc* d);
size_t conv3d_tcf_packed_bytes(const damvs_conv3d_desc* d);
int conv3d_tcf_pack(const damvs_conv3d_desc* d, const float* weight, void* packed, cudaStream_t st);
// prob layer (8 -> 1, plain fp32 output): every tap folded into N (conv3d_tcp.cu)
bool conv3d_tcp_supported(const damvs_conv3d_desc* d);
size_t conv3d_tcp_packed_bytes(const damvs_conv3d_desc* d);
int conv3d_tcp_pack(const damvs_conv3d_desc* d, const float* weight, void* packed, cudaStream_t st);
int conv3d_tcp_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, void* out, cudaStream_t st);
int conv3d_tcf_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, const float* scale, const float* shift,
                      const void* skip, void* out, cudaStream_t st);

// how many output-channel blobs a layer is split into so that weights + ring fit in shared memory
static int n_split(int Cin, int Cout) { return (Cin >= 64 && Cout >= 64) ? 2 : 1; }

static size_t blob_bytes(int nsteps, int CP) { return (size_t)weights_offset(nsteps) + (size_t)nsteps * 2 * 3 * CP * 16; }

size_t conv3d_tc_packed_bytes(const damvs_conv3d_desc* d) {
  if (conv3d_tcp_supported(d)) return conv3d_tcp_packed_bytes(d) + conv3d_tcf_packed_bytes(d);   // odd depths use the depth-folded kernel
  if (conv3d_tcf_supported(d)) return conv3d_tcf_packed_bytes(d);
  std::vector<StepSrc> steps;
  if (!build_program(mode_of(d), d->Cin / 8, steps)) return 0;
  int split = n_split(d->Cin, d->Cout);
  int CP = padded_c(d->Cout / split);
  return (blob_bytes((int)steps.size(), CP) + 255) / 256 * 256 * split;
}

// B operand of step s: [2 K-halves][N = 3*CP rows][8 channels] bf16; row n = j*CP + co where j is the folded
// w tap (conv: kw = j; transposed: tw = {1, 2, 0}[j]).
// The header and the step table travel as a by-value kernel argument and are written by the kernel itself: packing is
// fully asynchronous (no staging copy, no stream synchronisation), so it can run every training step and inside graphs.
struct PackMeta {
  PackedHeader hdr;
  StepSrc steps[kMaxSteps];
};
__global__ void pack_weight_tc_kernel(const float* __restrict__ w, uint8_t* __restrict__ blob, const __grid_constant__ PackMeta meta, int Cin,
                                      int Cout, int co_end, int transposed, int CP, int n0, int nsteps, int f16) {
  uint16_t* dst = reinterpret_cast<uint16_t*>(blob + weights_offset(nsteps));
  const int N = 3 * CP;
  int i = blockIdx.x * blockDim.x + threadIdx.x;  // over [nsteps][2][N][8]
  if (i == 0) *reinterpret_cast<PackedHeader*>(blob) = meta.hdr;
  if (i < nsteps) reinterpret_cast<StepSrc*>(blob + steps_offset())[i] = meta.steps[i];
  if (i >= nsteps * 2 * N * 8) return;
  int j8 = i & 7, n = (i >> 3) % N, h = (i / (8 * N)) & 1, s = i / (16 * N);
  StepSrc st = meta.steps[s];
  const int jw = n / CP, col = n - jw * CP;
  const int kw = transposed ? (jw == 0 ? 1 : (jw == 1 ? 2 : 0)) : jw;
  int co = n0 + col, ci = st.g[h] * 8 + j8, tap2 = st.tap[h];
  float v = 0.f;
  if (tap2 >= 0 && co < co_end) {
    const int tap = tap2 * 3 + kw;
    v = transposed ? w[((size_t)ci * Cout + co) * 27 + tap] : w[((size_t)co * Cin + ci) * 27 + tap];
  }
  dst[i] = f16 ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
}

int conv3d_tc_pack(const damvs_conv3d_desc* d, const float* weight, void* packed, cudaStream_t st) {
  if (conv3d_tcp_supported(d)) {
    const int rc = conv3d_tcp_pack(d, weight, packed, st);
    return rc != DAMVS_OK ? rc : conv3d_tcf_pack(d, weight, (uint8_t*)packed + conv3d_tcp_packed_bytes(d), st);
  }
  if (conv3d_tcf_supported(d)) return conv3d_tcf_pack(d, weight, packed, st);
  std::vector<StepSrc> steps;
  const int mode = mode_of(d), G = d->Cin / 8;
  if (!build_program(mode, G, steps)) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: Cin=%d not supported", d->Cin);
  if (d->Cout > 64 && !d->plain_out) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: Cout=%d > 64", d->Cout);
  const int split = n_split(d->Cin, d->Cout);
  const int cper = d->Cout / split;
  const int CP = padded_c(cper);
  const int nsteps = (int)steps.size();
  const size_t bb = (blob_bytes(nsteps, CP) + 255) / 256 * 256;
  for (int k = 0; k < split; ++k) {
    uint8_t* blob = (uint8_t*)packed + k * bb;
    PackMeta meta{};
    PackedHeader& h = meta.hdr;
    h.magic = kMagic; h.mode = mode; h.Cin = d->Cin; h.Cout = d->Cout; h.CP = CP; h.nsteps = nsteps;
    h.ncls = mode == MODE_T ? 4 : 1; h.n0 = k * cper; h.blob_bytes = (int)bb; h.nblobs = split; h.f16 = d->in_dtype == DAMVS_F16 ? 1 : 0;
    for (int i = 0; i < nsteps; ++i) meta.steps[i] = steps[i];
    int total = nsteps * 2 * 3 * CP * 8;
    // the blob computes channels [n0, n0 + cper); rows beyond that are zero padding
    pack_weight_tc_kernel<<<(total + 255) / 256, 256, 0, st>>>(weight, blob, meta, d->Cin, d->Cout, (k + 1) * cper, d->transposed, CP,
                                                              k * cper, nsteps, d->in_dtype == DAMVS_F16 ? 1 : 0);
    DAMVS_LAUNCH_OK("pack_weight_tc kernel");
  }
  return DAMVS_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

// G8 bf16 volume [BG][D][H][W*8] viewed with rows (row0, row0 + row_step, ...)
static int make_map(CUtensorMap* m, const void* base, int BG, int D, int H, int W, int row0, int row_step, int box_rows, int G, bool f16) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(DAMVS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  const int nrows = (H - row0 + row_step - 1) / row_step;
  cuuint64_t dims[4] = {(cuuint64_t)W * 8, (cuuint64_t)(nrows > 0 ? nrows : 1), (cuuint64_t)D, (cuuint64_t)BG};
  cuuint64_t strides[3] = {(cuuint64_t)W * 16 * row_step, (cuuint64_t)H * W * 16, (cuuint64_t)D * H * W * 16};
  cuuint32_t box[4] = {(cuuint32_t)kP * 8, (cuuint32_t)box_rows, 1, (cuuint32_t)G};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  void* addr = (void*)((const uint8_t*)base + (size_t)row0 * W * 16);
  CUresult r = fn(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, addr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(DAMVS_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) W=%d H=%d D=%d BG=%d rows=%d", (int)r, W, H, D, BG, box_rows);
  return DAMVS_OK;
}

static size_t slot_bytes(int mode, int G, int MC) {
  const int rows = mode == MODE_S1 ? 4 * MC + 2 : (mode == MODE_T ? 4 * MC + 1 : 8 * MC + 1);
  return (size_t)G * rows * kP * 16;
}
static size_t fixed_smem(int CP, int nsteps) {
  return (size_t)nsteps * 2 * 3 * CP * 16 + 2 * CP * sizeof(float) + (2 * kMaxSlots + 5) * sizeof(uint64_t) + 16;
}
constexpr size_t kSmemBudget = 227 * 1024;
// at most 8 planes in the ring (the TMA runs up to 8 - span planes ahead): a deeper ring only takes shared memory from
// co-resident CTAs
constexpr int kSlotCap = 8;
static_assert(kSlotCap <= kMaxSlots, "barrier arrays hold kMaxSlots slots");

template <int MODE, int CP, int MC, int G, bool F16>
static int launch_one(const damvs_conv3d_desc* d, TcParams& P, const void* in, const std::vector<StepSrc>& steps, cudaStream_t st) {
  using G_ = Geo<MODE>;
  const int nsteps = (int)steps.size();
  P.nsteps = nsteps;
  CUtensorMap m0, m1;
  int rc;
  if (MODE == MODE_S2) {
    if ((rc = make_map(&m0, in, d->B * G, d->Din, d->Hin, d->Win, 0, 2, G_::rows0(MC), G, F16))) return rc;
    if ((rc = make_map(&m1, in, d->B * G, d->Din, d->Hin, d->Win, 1, 2, G_::rows1(MC), G, F16))) return rc;
  } else {
    if ((rc = make_map(&m0, in, d->B * G, d->Din, d->Hin, d->Win, 0, 1, G_::rows0(MC), G, F16))) return rc;
    m1 = m0;
  }
  // ring depth: TMA runs ahead of the MMAs by nslots - span planes
  const size_t sb = slot_bytes(MODE, G, MC), fx = fixed_smem(CP, nsteps);
  int nslots = std::min((int)((kSmemBudget - fx) / sb), kSlotCap);
  if (nslots < G_::span + 1) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: ring does not fit");
  // leave room for a second CTA per SM when a deep ring is not needed
  while (nslots > G_::span + 1 && fx + (size_t)nslots * sb + 1024 > kSmemBudget / 2) --nslots;
  P.nslots = nslots;
  const size_t smem = fx + (size_t)nslots * sb;
  auto kern = conv3d_tc_kernel<MODE, CP, MC, G, F16>;
  DAMVS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int TH = 4 * MC;
  const int tiles_h = MODE == MODE_T ? d->Hin : P.Hout, tiles_w = MODE == MODE_T ? d->Win : P.Wout;
  P.tiles_x = (tiles_w + G_::TW - 1) / G_::TW;
  P.tiles_y = (tiles_h + TH - 1) / TH;
  // very few spatial tiles (the bottleneck level of stage 1): split the depth range so that more SMs get work; each
  // chunk re-loads span - adv halo planes.  Measured: splitting every layer with < 2 tiles per SM helps one view in
  // flight (3.54 -> 3.48 ms) and costs throughput with 3-4 views in flight (more CTAs contending), hence the low bar.
  {
    const int spatial = P.tiles_x * P.tiles_y * d->B;
    int zc = 1;
    if (spatial * 2 < 148) {
      const int want = (148 + spatial - 1) / spatial;
      const int min_len = spatial * 4 < 148 ? 1 : 2;
      zc = std::max(1, std::min(want, P.niter / min_len));
    }
    P.zlen = (P.niter + zc - 1) / zc;
    P.zchunks = (P.niter + P.zlen - 1) / P.zlen;
    P.ntiles = spatial * P.zchunks;
  }
  // persistent grid: as many CTAs as fit at once (shared memory, TMEM columns, registers)
  DAMVS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  cudaFuncAttributes fa;
  DAMVS_CUDA_OK(cudaFuncGetAttributes(&fa, kern));
  const int regs_per_cta = ((fa.numRegs + 7) / 8 * 8) * 320;
  int occ = std::min({(int)((228 * 1024) / (smem + fa.sharedSizeBytes + 1024)), 65536 / regs_per_cta, 2048 / 320});
  constexpr int ACC = Geo<MODE>::ncls * MC * 3 * CP;
  constexpr int NEEDC = nbuf_of(MODE, CP, ACC) * ACC;
  constexpr int TCOLS = NEEDC <= 32 ? 32 : NEEDC <= 64 ? 64 : NEEDC <= 128 ? 128 : NEEDC <= 256 ? 256 : 512;
  occ = std::max(1, std::min(occ, 512 / TCOLS));
  dim3 grid((unsigned)std::min(P.ntiles, occ * current_sm_count()), 1, 1);
  kern<<<grid, 320, smem, st>>>(m0, m1, P);
  DAMVS_LAUNCH_OK("conv3d_tc kernel");
  return DAMVS_OK;
}

static bool mc_fits(int mode, int G, int CP, int nsteps, int mc) {
  const int ncls = mode == MODE_T ? 4 : 1, span = mode == MODE_T ? 2 : 3;
  const int acc = ncls * mc * 3 * CP;
  if (acc > 512) return false;
  // taller tiles only while the double-buffered accumulator stays within 256 TMEM columns (two CTAs per SM)
  if (mc > 1 && 2 * acc > 256) return false;
  return fixed_smem(CP, nsteps) + (size_t)(span + 1) * slot_bytes(mode, G, mc) <= kSmemBudget;
}

// tile height (4*MC rows): the largest that fits shared memory / TMEM and still yields >= 2 CTAs per SM;
// when there is not enough work for that at any height, the smallest tile (most CTAs)
static int pick_mc(int mode, int G, int CP, int nsteps, int tile_rows, int tile_cols, int B) {
  const int TW = mode == MODE_S1 ? 30 : (mode == MODE_T ? 31 : 15);
  for (int mc = 4; mc >= 1; mc >>= 1) {
    if (!mc_fits(mode, G, CP, nsteps, mc)) continue;
    const long long ctas = (long long)((tile_cols + TW - 1) / TW) * ((tile_rows + 4 * mc - 1) / (4 * mc)) * B;
    if (ctas >= 2 * 148) return mc;
  }
  for (int mc = 1; mc <= 4; mc <<= 1)
    if (mc_fits(mode, G, CP, nsteps, mc)) return mc;
  return 0;
}

int conv3d_tc_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, const float* scale, const float* shift,
                     const void* skip, void* out, cudaStream_t st) {
  if ((d->in_dtype != DAMVS_BF16 && d->in_dtype != DAMVS_F16) || (!d->plain_out && d->out_dtype != d->in_dtype))
    return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: bf16 or fp16 volumes only (input and output of the same type)");
  const bool f16 = d->in_dtype == DAMVS_F16;
  if (d->plain_out && (d->transposed || d->stride != 1)) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: plain_out is stride-1 only");
  if (conv3d_tcp_supported(d)) {
    if (d->Din % 2 == 0) return conv3d_tcp_launch(d, in, packed, out, st);
    return conv3d_tcf_launch(d, in, (const uint8_t*)packed + conv3d_tcp_packed_bytes(d), scale, shift, skip, out, st);
  }
  if (conv3d_tcf_supported(d)) return conv3d_tcf_launch(d, in, packed, scale, shift, skip, out, st);
  const int mode = mode_of(d), G = d->Cin / 8;
  if (G != 1 && G % 2) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: Cin=%d not supported", d->Cin);
  if (d->Cout > 64) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: Cout=%d > 64", d->Cout);
  if (mode == MODE_S2 && ((d->Hin & 1) || (d->Win & 1) || (d->Din & 1)))
    return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: stride-2 needs even input extents");
  const int split = n_split(d->Cin, d->Cout);
  const int cper = d->Cout / split;
  const int CP = padded_c(cper);
  if (mode == MODE_T && CP > 32) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: transposed Cout=%d > 32", d->Cout);
  TcParams P{};
  P.scale = scale; P.shift = shift; P.skip = (const uint16_t*)skip; P.out = out;
  P.B = d->B; P.G = G; P.Din = d->Din; P.Hin = d->Hin; P.Win = d->Win;
  if (d->transposed) { P.Dout = 2 * d->Din; P.Hout = 2 * d->Hin; P.Wout = 2 * d->Win; P.niter = d->Din; }
  else { P.Dout = (d->Din - 1) / d->stride + 1; P.Hout = (d->Hin - 1) / d->stride + 1; P.Wout = (d->Win - 1) / d->stride + 1; P.niter = P.Dout; }
  P.out_G = d->plain_out ? 1 : d->Cout / 8; P.relu = d->relu; P.plain_out = d->plain_out;
  std::vector<StepSrc> steps;
  if (!build_program(mode, G, steps)) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: no program for Cin=%d", d->Cin);
  const int nsteps = (int)steps.size();
  const size_t bb = (blob_bytes(nsteps, CP) + 255) / 256 * 256;
  const int mc = pick_mc(mode, G, CP, nsteps, mode == MODE_T ? d->Hin : P.Hout, mode == MODE_T ? d->Win : P.Wout, d->B);
  if (mc == 0) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: Cin=%d Cout=%d does not fit in shared memory", d->Cin, d->Cout);
  for (int k = 0; k < split; ++k) {
    P.blob = (const uint8_t*)packed + k * bb;
    P.n0 = k * cper; P.out_g0 = (k * cper) / 8; P.Cout = d->plain_out ? 1 : (k + 1) * cper;
    int rc = -1;
#define GO(MODE_, CP_, MC_, G_)                                   \
  if (mode == MODE_ && CP == CP_ && mc == MC_ && G == G_)         \
    rc = f16 ? launch_one<MODE_, CP_, MC_, G_, true>(d, P, in, steps, st) : launch_one<MODE_, CP_, MC_, G_, false>(d, P, in, steps, st)
    // the layer shapes of CostRegNet with base_channels 8 (reference models/module.py:513-530); stride-1 layers with
    // Cout <= 16 (conv0, conv2, prob) run on conv3d_tcf.cu / conv3d_tcp.cu
    GO(MODE_S1, 32, 1, 4);                           // conv4
    GO(MODE_S1, 32, 1, 1);                           // adjoint of conv0 (stage 1): 8 -> 32
    GO(MODE_S1, 32, 1, 8);                           // conv6 (two output halves)
    GO(MODE_S2, 16, 2, 1); GO(MODE_S2, 16, 1, 1);   // conv1
    GO(MODE_S2, 32, 1, 2);                           // conv3
    GO(MODE_S2, 64, 1, 4);                           // conv5
    GO(MODE_T, 32, 1, 8);                            // conv7
    GO(MODE_T, 16, 2, 4); GO(MODE_T, 16, 1, 4);     // conv9
    GO(MODE_T, 16, 2, 2); GO(MODE_T, 16, 1, 2);     // conv11
#undef GO
    if (rc == -1) return set_error(DAMVS_ERR_UNSUPPORTED, "conv3d tcgen05: no kernel for mode=%d Cin=%d CP=%d MC=%d", mode, d->Cin, CP, mc);
    if (rc) return rc;
  }
  return DAMVS_OK;
}

}  // namespace damvs
