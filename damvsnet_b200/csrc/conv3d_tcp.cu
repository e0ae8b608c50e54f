// tcgen05 / TMEM kernel for the `prob` layer (8 channels -> 1 logit, 3x3x3, stride 1, no bias, fp32 [B, D, H, W] output;
// reference models/module.py:530, consumed by the softmax head).
//
// With a single output channel every filter tap can be a column of N.  One MMA per PAIR of input planes computes
//     Y[j][kh][kw][m] = sum_{half, ci} in_{2i+half}[m][ci] * W[kd(j, half), kh, kw][ci]       K = 2 planes x 8 channels
// for the four output planes z = 2i - 1 + j that the pair touches (N = 4 x 16 columns, 9 of each 16 used), where m is
// an input position of the tile.  The A operand -- the 4 KB shared-memory read that bounds the MMA rate of the
// small-N kernels (DESIGN.md section 3.2) -- is read once per plane pair instead of 2 (kh steps) x 1.5 (ring wrap)
// times per plane: a sixth of the depth-folded kernel's MMA time (conv3d_tcf.cu), which is what that kernel was
// bound by on this layer.  The output-plane accumulators live in a ring of eight 16-column TMEM slots per 128-row
// chunk; a window of four consecutive slots advances by two per iteration (split into two MMAs when it wraps).
//
// The taps are recombined in the epilogue, one output voxel per thread: kw by two shuffles per kh (lanes are x), kh by
// an exchange through shared memory between the warps of a half (rows are warps).  The tile is 8 x 32 input
// positions -> 6 x 30 outputs.  Slots are zeroed by the epilogue after draining, so every MMA accumulates.
//
// Warp roles (320 threads): warp 0 TMA producer, warp 1 MMA issuer (one thread), warps 2-9 epilogue in two groups of
// four; group g drains the output planes with global index = g mod 2, so the two planes an iteration completes are
// drained concurrently (four groups / 16 epilogue warps measured slower: their barrier spinning takes issue slots from
// the issuer).  Measured (phase knock-out experiments, DESIGN.md section 3.2): the issuer's instruction
// path per iteration is what bounds these kernels once the A reads are gone, hence one wait for the planes, one for
// the accumulator pair, at most four MMAs and ONE commit per iteration (the same barrier frees the shared-memory slot
// for the producer and publishes the completed output planes to the epilogue).
#include <algorithm>
#include <mutex>

#include "common.cuh"
#include "tc_common.cuh"

namespace damvs {

using namespace tc;

namespace tcp {

constexpr int kP = 32;           // patch pitch in voxels (one TMA box row = 32 voxels * 16 B)
constexpr int R0 = 8;            // patch rows = GEMM rows / 32
constexpr int TH = 6, TW = 30;   // outputs per tile
constexpr int MC = 2;            // 128-row chunks
constexpr int NBP = 16;          // accumulator columns per output plane (kh * 3 + kw; 9 used)
constexpr int RING = 8;          // accumulator slots per chunk
constexpr int WIN = 4;           // output planes one plane pair contributes to
constexpr int TMEM_COLS = MC * RING * NBP;   // 256: two CTAs per SM
constexpr int LOG_NS = 2, NS = 1 << LOG_NS;   // plane-pair slots in shared memory (deeper rings measured no faster; a small footprint
                                             // leaves room for the CTAs of the other views' kernels, DESIGN.md section 4)
constexpr int SLOT_BYTES = 2 * R0 * kP * 16; // two planes
constexpr int B_ROWS = WIN * NBP;            // 64
constexpr uint32_t kMagicP = 0x50435444u;    // "DTCP"

struct Header {  // 64 bytes
  uint32_t magic;
  int32_t Cin, pad[14];
};

struct Params {
  const uint8_t* blob;
  float* out;
  int B, D, H, W;
  int tiles_x, tiles_y, ntiles;
  uint32_t fmt_xor;   // 0 for bf16 operands; the A / B format bits of the instruction descriptor for fp16 (XOR turns them off)
  // fused head (HEAD = true): per-pixel hypotheses in, probability volume and the three maps out; `out` is unused
  const float* hyp;
  float* prob;
  float* depth;
  float* conf;
  float* var;
};

__device__ __forceinline__ float shfl_dn(uint32_t v, int d) { return __uint_as_float(__shfl_down_sync(0xffffffffu, v, d)); }
constexpr size_t kSmemBase = 45 * 1024;   // offset of the fused head's logits buffer (>= the base kernel's footprint)
constexpr int NG = 2;            // epilogue groups of four warps; group g drains the output planes with global index = g mod NG
constexpr int THREADS = 64 + NG * 128;
__device__ __forceinline__ void group_barrier(int g) {   // constant ids: a register id would reserve all 16 barriers
  if (g == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
  else if (g == 1) asm volatile("bar.sync 2, 128;" ::: "memory");
  else if (g == 2) asm volatile("bar.sync 3, 128;" ::: "memory");
  else asm volatile("bar.sync 4, 128;" ::: "memory");
}

// exp(x), x <= 0, argument clamped at -80: keeps e and e / s out of the denormal slow paths (see head.cu)
__device__ __forceinline__ float exp_clamped_p(float x) { return expf(x < -80.f ? -80.f : x); }   // NaN propagates (head.cu)

// HEAD = true fuses the softmax / regression / confidence / variance head (head.cu; reference models/cas_mvsnet.py:105-124)
// into the epilogue: the CTA owns all D output planes of its 6 x 30 pixels, so the logits go to shared memory ([D][8][32]
// fp32) instead of HBM, and when a tile's last plane has been drained the eight epilogue warps turn into a one-thread-per-
// pixel head (same arithmetic as head_reg_kernel) that reads the pixel's hypothesis column (prefetched into L2 at the start
// of the tile), writes prob_volume and the three maps, and hands the buffer back.  The logits never reach HBM (2 x D*h*w*4
// bytes and one launch per stage saved); the MMA / TMA warps keep running up to RING planes ahead meanwhile.
template <bool HEAD>
__global__ void __launch_bounds__(THREADS, 2) conv3d_tcp_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ Params P) {
  constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);   // SBO = 128 B, descriptor version 1
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;
  uint8_t* sB = sA + NS * SLOT_BYTES;                    // [2 planes][64 rows][16 B]
  float* sX = reinterpret_cast<float*>(sB + 2 * B_ROWS * 16); // kh exchange: [group][buffer][row 8][kh 1..2][32]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sX + NG * 2 * R0 * 2 * 32);
  uint64_t* full = bars;              // TMA -> MMA: plane pair landed
  uint64_t* done = bars + NS;         // MMA -> TMA and epilogue: the iteration's MMAs have completed
  uint64_t* acc_empty = bars + 2 * NS; // epilogue -> MMA: a pair of accumulator slots drained and zeroed (8 warps)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + RING / 2);
  float* sL = reinterpret_cast<float*>(smem + kSmemBase);   // HEAD: logits / probabilities of the tile, [D][8 rows][32]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Header* hdr = reinterpret_cast<const Header*>(P.blob);
  if (hdr->magic != kMagicP || hdr->pad[0] != (P.fmt_xor ? 1 : 0)) {   // wrong layer type, or weights packed for the other 2-byte format
    if (threadIdx.x == 0 && blockIdx.x == 0) printf("damvs: packed conv weights were not built for the prob kernel\n");
    __trap();
  }
  {
    const uint4* wsrc = reinterpret_cast<const uint4*>(P.blob + sizeof(Header));
    uint4* wdst = reinterpret_cast<uint4*>(sB);
    for (int i = threadIdx.x; i < 2 * B_ROWS; i += blockDim.x) wdst[i] = __ldg(wsrc + i);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&full[i], 1); mbar_init(&done[i], 1); }
    for (int i = 0; i < RING / 2; ++i) mbar_init(&acc_empty[i], 8);
    fence_barrier_init();
    tma_prefetch_desc(&map0);
  }
  if (warp == 1) tmem_alloc(tmem_ptr, TMEM_COLS);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int D = P.D, NIT = D / 2;   // D is even (conv3d_tcp_supported)
#define TILE_COORDS(tile_)                                   \
  const int b = (int)((uint32_t)(tile_) / (uint32_t)(P.tiles_x * P.tiles_y));                               \
  const int ty0 = (int)(((uint32_t)(tile_) / (uint32_t)P.tiles_x) % (uint32_t)P.tiles_y) * TH;               \
  const int tx0 = (int)((uint32_t)(tile_) % (uint32_t)P.tiles_x) * TW;

  if (warp == 0) {
    // ===== TMA producer: two input planes per iteration =====
    if (lane == 0) {
      uint32_t gi = 0;
      for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
        TILE_COORDS(tile)
        for (int i = 0; i < NIT; ++i, ++gi) {
          const uint32_t slot = gi & (NS - 1);
          if (gi >= NS) mbar_wait(&done[slot], ((gi >> LOG_NS) - 1) & 1u);
          mbar_arrive_expect_tx(&full[slot], (uint32_t)SLOT_BYTES);
          tma_load_4d(sA + slot * SLOT_BYTES, &map0, &full[slot], (tx0 - 1) * 8, ty0 - 1, 2 * i, b);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: one thread; per iteration one wait for the planes, one for the accumulators, <= 4 MMAs, one commit =====
    if (lane == 0) {
      const uint32_t a_base16 = smem_u32(sA) >> 4, b_base16 = smem_u32(sB) >> 4;
      uint32_t gi = 0;   // iterations issued by this CTA
      uint32_t zb = 0;   // output planes produced by this CTA before the current tile (ring position of its plane 0; even)
      for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x, zb += D) {
        for (int i = 0; i < NIT; ++i, ++gi) {
          const uint32_t slot = gi & (NS - 1);
          mbar_wait(&full[slot], (gi >> LOG_NS) & 1u);
          // planes 2i + 1 and 2i + 2 get their first contribution now: their slots (pair m) must have been drained
          const uint32_t m = (zb >> 1) + i + 1;
          if (m >= RING / 2) mbar_wait(&acc_empty[m & (RING / 2 - 1)], ((m >> 2) - 1) & 1u);
          tc_fence_after();
          // Column blocks j = 0..3 <-> output plane 2i - 1 + j.  Planes 2i - 1, 2i (accumulator pair m - 1) already hold the
          // earlier planes' contributions; planes 2i + 1, 2i + 2 (pair m) are written for the first time, which the MMA's
          // accumulate flag expresses -- nothing is ever zeroed.  Plane g lives in slot (g + 1) mod 8, so a pair never
          // straddles the end of the ring.
          const uint32_t alo = (a_base16 + slot * (SLOT_BYTES >> 4)) | ((uint32_t)(R0 * kP) << 16);   // LBO = one plane
          const uint32_t blo = b_base16 | ((uint32_t)B_ROWS << 16);                                     // LBO = 64 rows * 16 B
          const uint32_t d_old = tmem_base + ((m - 1) & (RING / 2 - 1)) * (2 * NBP), d_new = tmem_base + (m & (RING / 2 - 1)) * (2 * NBP);
          const bool first = i == 0, last = i == NIT - 1;
#pragma unroll
          for (int c = 0; c < MC; ++c) {
            const uint64_t adesc = ((uint64_t)DESC_HI << 32) | (alo + c * 128);
            // a tile's first pair only touches plane 0 (block 1), and starts it
            mma_bf16_ss(d_old + c * (RING * NBP) + (first ? NBP : 0), adesc, ((uint64_t)DESC_HI << 32) | (blo + (first ? NBP : 0)),
                        idesc_bf16_m128(first ? NBP : 2 * NBP) ^ P.fmt_xor, first ? 0u : 1u);
            // its last pair only touches plane D - 1 (block 2)
            mma_bf16_ss(d_new + c * (RING * NBP), adesc, ((uint64_t)DESC_HI << 32) | (blo + 2 * NBP), idesc_bf16_m128(last ? NBP : 2 * NBP) ^ P.fmt_xor, 0u);
          }
          mma_commit(&done[slot]);   // the plane pair can be overwritten; output planes 2i - 1, 2i (and D - 1 at the end) are complete
        }
      }
    }
  } else {
    // ===== epilogue: warp (q, grp) owns patch rows q and 4 + q of the output planes with global index = grp mod NG =====
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const size_t HW = (size_t)P.H * P.W;
    float* xbase = sX + grp * (2 * R0 * 2 * 32) + q * 64 + lane;   // row q, kh 1
    const uint32_t tq = tmem_base + ((uint32_t)(32 * q) << 16);
    int buf = 0;
    uint32_t zb = 0, gib = 0;
    if (grp == NG - 1 && lane == 0) mbar_arrive(&acc_empty[0]);   // stands in for the plane before the first one
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x, zb += D, gib += NIT) {
      TILE_COORDS(tile)
      const int z0 = (int)((grp - zb) & (NG - 1));   // first plane of this tile that belongs to the group
      bool valid[MC];
      float* op[MC];
#pragma unroll
      for (int c = 0; c < MC; ++c) {
        const int pr = c * 4 + q, yo = ty0 + pr, xo = tx0 + lane;
        valid[c] = pr < TH && lane < TW && yo < P.H && xo < P.W;
        op[c] = P.out + ((size_t)b * D + z0) * HW + (size_t)yo * P.W + xo;
      }
      if (HEAD) {
        // pull the tile's hypothesis columns into L2 while the planes are being computed: warp w <-> tile row w,
        // lane <-> plane (two lanes per 32 planes cover the first and the last byte of the row's 120-byte segment)
        const int wi = grp * 4 + q;
        if (wi < TH && ty0 + wi < P.H) {
          const float* hrow = P.hyp + ((size_t)b * D) * HW + (size_t)(ty0 + wi) * P.W;
          const int xa = tx0, xe = min(tx0 + TW, P.W) - 1;
          for (int k = lane; k < D; k += 32) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(hrow + (size_t)k * HW + xa));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(hrow + (size_t)k * HW + xe));
          }
        }
      }
      for (int z = z0; z < D; z += NG) {
        const uint32_t gz = zb + z;
        const int sl = (int)((gz + 1) & (RING - 1));
        const uint32_t g = gib + min((z + 1) >> 1, NIT - 1);   // the iteration that completes plane z
        mbar_wait(&done[g & (NS - 1)], (g >> LOG_NS) & 1u);
        tc_fence_after();
        const uint32_t pair = ((gz + 1) >> 1) & (RING / 2 - 1);
        uint32_t y[MC][8], y8[MC];   // taps kh * 3 + kw = 0..7 and 8
#pragma unroll
        for (int c = 0; c < MC; ++c) {
          const uint32_t tbase = tq + (c * RING + sl) * NBP;
          tmem_ld8(tbase, y[c]);
          tmem_ld1(tbase + 8, y8[c]);
        }
        tmem_ld_wait();
        tc_fence_before();
        if (lane == 0) mbar_arrive(&acc_empty[pair]);   // the slot has been read: hand it back
        float u0[MC];
        float* xb = xbase + buf * (R0 * 2 * 32);
#pragma unroll
        for (int c = 0; c < MC; ++c) {
          u0[c] = __uint_as_float(y[c][0]) + shfl_dn(y[c][1], 1) + shfl_dn(y[c][2], 2);
          const float u1 = __uint_as_float(y[c][3]) + shfl_dn(y[c][4], 1) + shfl_dn(y[c][5], 2);
          const float u2 = __uint_as_float(y[c][6]) + shfl_dn(y[c][7], 1) + shfl_dn(y8[c], 2);
          xb[c * 256] = u1;
          xb[c * 256 + 32] = u2;
        }
        group_barrier(grp);
#pragma unroll
        for (int c = 0; c < MC; ++c) {
          // kh 1 of the next row, kh 2 of the one after; patch rows 6, 7 have no output (and nothing to read beyond them)
          if (HEAD) {
            if (c * 4 + q < TH) sL[(z * 8 + c * 4 + q) * 32 + lane] = u0[c] + xb[c * 256 + 64] + xb[c * 256 + 128 + 32];
          } else {
            if (valid[c]) *op[c] = u0[c] + xb[c * 256 + 64] + xb[c * 256 + 128 + 32];
            op[c] += (size_t)NG * HW;
          }
        }
        buf ^= 1;
      }
      if (HEAD) {
        asm volatile("bar.sync 5, 256;" ::: "memory");   // both groups: every logit of the tile is in shared memory
        const int wi = grp * 4 + q, yo = ty0 + wi, xo = tx0 + lane;
        if (wi < TH && lane < TW && yo < P.H && xo < P.W) {
          float* col = sL + wi * 32 + lane;               // element k at col[k * 256]
          const size_t pix = (size_t)yo * P.W + xo;
          const float* hp = P.hyp + ((size_t)b * D) * HW + pix;
          float m = -INFINITY;
          for (int k = 0; k < D; ++k) m = fmaxf(m, col[k * 256]);
          float s = 0.f;
          for (int k = 0; k < D; ++k) {
            const float e = exp_clamped_p(col[k * 256] - m);
            col[k * 256] = e;
            s += e;
          }
          const float inv_s = 1.f / s;
          float dsum = 0.f, isum = 0.f;
          float* pr = P.prob + ((size_t)b * D) * HW + pix;
          for (int k0 = 0; k0 < D; k0 += 8) {             // D is a multiple of 8; eight independent loads in flight
            float h[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) h[j] = __ldg(hp + (size_t)(k0 + j) * HW);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float pk = col[(k0 + j) * 256] * inv_s;
              col[(k0 + j) * 256] = pk;
              dsum += pk * h[j];
              isum += pk * (float)(k0 + j);
              __stcs(pr + (size_t)(k0 + j) * HW, pk);
            }
          }
          float d2sum = 0.f;
          for (int k0 = 0; k0 < D; k0 += 8) {
            float h[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) h[j] = __ldg(hp + (size_t)(k0 + j) * HW);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float df = h[j] - dsum;
              d2sum += (df * df) * col[(k0 + j) * 256];
            }
          }
          long long idx = (long long)isum;                // .long() truncation, reference cas_mvsnet.py:116
          idx = idx < 0 ? 0 : (idx > D - 1 ? D - 1 : idx);
          float cf = 0.f;
          for (int k = (int)idx - 1; k <= (int)idx + 2; ++k)
            if (k >= 0 && k < D) cf += col[k * 256];
          const size_t o = (size_t)b * HW + pix;
          P.depth[o] = dsum;
          P.conf[o] = cf;
          P.var[o] = 3.f * sqrtf(d2sum);
        }
        asm volatile("bar.sync 5, 256;" ::: "memory");   // the buffer may be overwritten by the next tile's planes
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

// B operand: [2 planes of the pair][64 rows][8 channels] bf16; row n = j * 16 + kh * 3 + kw for output plane 2i - 1 + j,
// whose depth tap is kd = 2 - j for the first plane of the pair and 3 - j for the second.
__global__ void pack_weight_tcp_kernel(const float* __restrict__ w, uint8_t* __restrict__ blob, const __grid_constant__ Header hdr) {
  uint16_t* dst = reinterpret_cast<uint16_t*>(blob + sizeof(Header));
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // over [2][64][8]
  if (i == 0) *reinterpret_cast<Header*>(blob) = hdr;
  if (i >= 2 * B_ROWS * 8) return;
  const int ci = i & 7, n = (i >> 3) % B_ROWS, hh = i / (8 * B_ROWS);
  const int j = n / NBP, t = n % NBP, kd = 2 + hh - j;
  float v = 0.f;
  if (t < 9 && kd >= 0 && kd < 3) v = w[(size_t)ci * 27 + kd * 9 + t];
  dst[i] = hdr.pad[0] ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
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

constexpr size_t kSmem = (size_t)NS * SLOT_BYTES + 2 * B_ROWS * 16 + NG * 2 * R0 * 2 * 32 * sizeof(float) + (2 * NS + RING / 2) * sizeof(uint64_t) + 16;
static_assert(kSmem <= kSmemBase, "the fused head's logits buffer starts at kSmemBase");
constexpr int kHeadMaxD = 64;   // D * 1 KB of logits per CTA: two CTAs per SM up to D = 64

}  // namespace tcp

// ---- entry points used by conv3d_tc.cu's dispatch ------------------------------------------------------------------
bool conv3d_tcp_supported(const damvs_conv3d_desc* d) {
  return d->plain_out && !d->transposed && d->stride == 1 && d->Cin == 8;   // the layer; odd depths are launched on conv3d_tcf.cu
}

size_t conv3d_tcp_packed_bytes(const damvs_conv3d_desc*) { return (sizeof(tcp::Header) + 2 * tcp::B_ROWS * 16 + 255) / 256 * 256; }

int conv3d_tcp_pack(const damvs_conv3d_desc* d, const float* weight, void* packed, cudaStream_t st) {
  tcp::Header h{};
  h.magic = tcp::kMagicP; h.Cin = d->Cin; h.pad[0] = d->in_dtype == DAMVS_F16 ? 1 : 0;
  const int total = 2 * tcp::B_ROWS * 8;
  tcp::pack_weight_tcp_kernel<<<(total + 255) / 256, 256, 0, st>>>(weight, (uint8_t*)packed, h);
  DAMVS_LAUNCH_OK("pack_weight_tcp kernel");
  return DAMVS_OK;
}

template <bool HEAD>
static int tcp_launch_impl(const damvs_conv3d_desc* d, const void* in, const void* packed, tcp::Params P, cudaStream_t st) {
  using namespace tcp;
  P.blob = (const uint8_t*)packed;
  P.B = d->B; P.D = d->Din; P.H = d->Hin; P.W = d->Win;
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(DAMVS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  CUtensorMap m0;
  cuuint64_t dims[4] = {(cuuint64_t)d->Win * 8, (cuuint64_t)d->Hin, (cuuint64_t)d->Din, (cuuint64_t)d->B};
  cuuint64_t strides[3] = {(cuuint64_t)d->Win * 16, (cuuint64_t)d->Hin * d->Win * 16, (cuuint64_t)d->Din * d->Hin * d->Win * 16};
  cuuint32_t box[4] = {(cuuint32_t)kP * 8, (cuuint32_t)R0, 2, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const bool f16 = d->in_dtype == DAMVS_F16;
  P.fmt_xor = f16 ? ((1u << 7) | (1u << 10)) : 0u;
  CUresult r = fn(&m0, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(in), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(DAMVS_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  const size_t smem = HEAD ? kSmemBase + (size_t)d->Din * 8 * 32 * sizeof(float) : kSmem;
  auto kern = conv3d_tcp_kernel<HEAD>;
  DAMVS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DAMVS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  P.tiles_x = (d->Win + TW - 1) / TW;
  P.tiles_y = (d->Hin + TH - 1) / TH;
  P.ntiles = P.tiles_x * P.tiles_y * d->B;
  dim3 grid((unsigned)std::min(P.ntiles, 2 * current_sm_count()), 1, 1);   // two CTAs per SM (__launch_bounds__)
  kern<<<grid, THREADS, smem, st>>>(m0, P);
  DAMVS_LAUNCH_OK(HEAD ? "conv3d_tcp kernel (fused head)" : "conv3d_tcp kernel");
  return DAMVS_OK;
}

int conv3d_tcp_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, void* out, cudaStream_t st) {
  tcp::Params P{};
  P.out = (float*)out;
  return tcp_launch_impl<false>(d, in, packed, P, st);
}

// prob convolution + softmax / regression / confidence / variance head in one launch (even D <= 64, D % 8 == 0)
bool conv3d_tcp_head_supported(const damvs_conv3d_desc* d) {
  return conv3d_tcp_supported(d) && d->Din % 8 == 0 && d->Din <= tcp::kHeadMaxD &&
         (d->in_dtype == DAMVS_BF16 || d->in_dtype == DAMVS_F16);
}

int conv3d_tcp_head_launch(const damvs_conv3d_desc* d, const void* in, const void* packed, const float* hyp, float* prob, float* depth,
                           float* conf, float* var, cudaStream_t st) {
  tcp::Params P{};
  P.hyp = hyp; P.prob = prob; P.depth = depth; P.conf = conf; P.var = var;
  return tcp_launch_impl<true>(d, in, packed, P, st);
}

}  // namespace damvs
