// Geometric-consistency filtering of one reference view against its source views, fused (SURVEY.md section 8f, rank 2:
// the downstream neighbour of the path).
//
// Replaces, per reference view, the numpy + cv2.remap code of reference filter/dypcd.py:98-159
// (reproject_with_depth, check_geometric_consistency) and the accumulation over source views in filter_depth
// (filter/dypcd.py:205-257): the reference builds ~40 full-resolution float64 temporaries per (ref, src) pair on
// one CPU core; here one thread owns one reference pixel, walks the source views, and keeps the nine dynamic masks'
// counters, the consistent-depth sum and the final vote in registers.  HBM traffic: the reference depth and the
// three confidence maps once, four gathered taps of every source depth map, four small outputs.
//
// Arithmetic follows numpy's promotions so that the thresholded masks agree: projections in float64, the casts to
// float32 where the reference has `.astype(np.float32)`, the relative depth test in float32.  cv2.remap
// (INTER_LINEAR, BORDER_CONSTANT 0) is restated from OpenCV's published algorithm (opencv-python 4.x,
// imgproc/imgwarp.cpp remapBilinear): coordinates are rounded to 1/32 pixel, weights are the float32 products of
// the tabulated 1-D weights, taps outside the image contribute the border value 0.
#include <cuda/atomic>

#include "common.cuh"

namespace damvs {

constexpr int kMaxFuseSrc = 10;   // masks exist for i = 2..10 (filter/dypcd.py:151), so dy_range - 1 <= 10

struct FuseParams {
  const float* depth_ref;
  const float* conf[3];            // stage 1, 2, 3 confidence at the reference depth map's resolution
  const float* depth_src[kMaxFuseSrc];
  // per source view, float64: M_rs = E_src inv(E_ref) rows 0-2 [12], K_src [9], inv(K_src) [9], M_sr = E_ref inv(E_src) rows 0-2 [12]
  double cam[kMaxFuseSrc][42];
  double kref_inv[9], kref[9];
  float conf_thr[3];
  double dist_base, rel_diff_base;
  float* depth_avg;
  uint8_t* photo_mask;
  uint8_t* geo_mask;
  uint8_t* final_mask;
  int n_src, H, W;
};

__device__ __forceinline__ float remap_bilinear(const float* __restrict__ img, int H, int W, float x, float y) {
  // cv::remap, CV_32FC1 maps, INTER_LINEAR: sx = cvRound(x * 32) (round half to even), 5 fractional bits
  const int sx = __float2int_rn(x * 32.f), sy = __float2int_rn(y * 32.f);
  const int ix = sx >> 5, iy = sy >> 5;
  const float fx = (float)(sx & 31) * (1.f / 32.f), fy = (float)(sy & 31) * (1.f / 32.f);
  const float w00 = (1.f - fx) * (1.f - fy), w01 = fx * (1.f - fy), w10 = (1.f - fx) * fy, w11 = fx * fy;
  auto tap = [&](int yy, int xx) -> float {
    return ((unsigned)xx < (unsigned)W && (unsigned)yy < (unsigned)H) ? __ldg(img + (long long)yy * W + xx) : 0.f;
  };
  return tap(iy, ix) * w00 + tap(iy, ix + 1) * w01 + tap(iy + 1, ix) * w10 + tap(iy + 1, ix + 1) * w11;
}

struct FusePixel {
  float depth_avg;
  bool photo, geo;
};

// The filter at reference pixel (x, y), pix = y * W + x.  Both kernels below call it, so the masks of
// damvs_geo_consistency_points are those of damvs_geo_consistency_fuse by construction.
__device__ __forceinline__ FusePixel fuse_pixel(const FuseParams& P, int x, int y, long long pix) {
  const float dref = __ldg(P.depth_ref + pix);
  // reference 3-D point: inv(K_ref) [x, y, 1]^T * depth   (float64, filter/dypcd.py:105-106)
  const double dx = (double)x * (double)dref, dy = (double)y * (double)dref, dz = (double)dref;
  const double X = P.kref_inv[0] * dx + P.kref_inv[1] * dy + P.kref_inv[2] * dz;
  const double Y = P.kref_inv[3] * dx + P.kref_inv[4] * dy + P.kref_inv[5] * dz;
  const double Z = P.kref_inv[6] * dx + P.kref_inv[7] * dy + P.kref_inv[8] * dz;
  int geo_sum = 0, sums[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) sums[i] = 0;
  float depth_sum = 0.f;
  for (int v = 0; v < P.n_src; ++v) {
    const double* c = P.cam[v];
    const double sxx = c[0] * X + c[1] * Y + c[2] * Z + c[3];
    const double syy = c[4] * X + c[5] * Y + c[6] * Z + c[7];
    const double szz = c[8] * X + c[9] * Y + c[10] * Z + c[11];
    const double* K = c + 12;
    const double kx = K[0] * sxx + K[1] * syy + K[2] * szz, ky = K[3] * sxx + K[4] * syy + K[5] * szz, kz = K[6] * sxx + K[7] * syy + K[8] * szz;
    const double u = kx / kz, w = ky / kz;                       // xy_src (float64)
    const float samp = remap_bilinear(P.depth_src[v], P.H, P.W, (float)u, (float)w);
    const double* Ki = c + 21;
    const double ax = u * (double)samp, ay = w * (double)samp, az = (double)samp;
    const double px = Ki[0] * ax + Ki[1] * ay + Ki[2] * az, py = Ki[3] * ax + Ki[4] * ay + Ki[5] * az, pz = Ki[6] * ax + Ki[7] * ay + Ki[8] * az;
    const double* M = c + 30;
    const double rx = M[0] * px + M[1] * py + M[2] * pz + M[3];
    const double ry = M[4] * px + M[5] * py + M[6] * pz + M[7];
    const double rz = M[8] * px + M[9] * py + M[10] * pz + M[11];
    float depth_rep = (float)rz;
    double qx = P.kref[0] * rx + P.kref[1] * ry + P.kref[2] * rz, qy = P.kref[3] * rx + P.kref[4] * ry + P.kref[5] * rz,
           qz = P.kref[6] * rx + P.kref[7] * ry + P.kref[8] * rz;
    if (qz == 0.0) qz += 0.00001;
    const float xr = (float)(qx / qz), yr = (float)(qy / qz);
    const double ex = (double)xr - (double)x, ey = (double)yr - (double)y;
    const double dist = sqrt(ex * ex + ey * ey);
    const float rel = fabsf(depth_rep - dref) / dref;            // float32, filter/dypcd.py:145-146
    bool last = false;
#pragma unroll
    for (int i = 2; i <= 10; ++i) {
      const bool m = dist < (double)i * P.dist_base && rel < (float)((double)i * P.rel_diff_base);
      sums[i - 2] += m ? 1 : 0;
      last = m;
    }
    geo_sum += last ? 1 : 0;
    depth_sum += last ? depth_rep : 0.f;                          // depth_reprojected[~mask] = 0
  }
  const int dy_range = P.n_src + 1;
  bool geo = geo_sum >= dy_range;
#pragma unroll
  for (int i = 2; i <= 10; ++i)
    if (i < dy_range) geo = geo || sums[i - 2] >= i;
  const bool photo = __ldg(P.conf[2] + pix) > P.conf_thr[2] && __ldg(P.conf[1] + pix) > P.conf_thr[1] && __ldg(P.conf[0] + pix) > P.conf_thr[0];
  return {(float)((double)(depth_sum + dref) / (double)(geo_sum + 1)), photo, geo};
}

__global__ void __launch_bounds__(128) geo_fuse_kernel(const __grid_constant__ FuseParams P) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= P.W) return;
  const long long pix = (long long)y * P.W + x;
  const FusePixel r = fuse_pixel(P, x, y, pix);
  P.depth_avg[pix] = r.depth_avg;
  P.photo_mask[pix] = r.photo;
  P.geo_mask[pix] = r.geo;
  P.final_mask[pix] = r.photo && r.geo;
}

// ---- the filter's points, compacted in row-major pixel order (filter/dypcd.py:281-299) --------------------------
// One CTA owns one tile: kPointsTile pixels of one row.  Tiles number row-major, so the order of tiles and of the
// lanes within one is the reference's np.nonzero order.  A single-pass decoupled look-back scan turns the per-tile
// point counts into output offsets: a tile takes its index from an atomic ticket (so every tile it waits for has
// already started and cannot be waiting for it), publishes its count, sums its predecessors' published words back to
// the nearest inclusive prefix, then publishes its own inclusive prefix.
constexpr int kPointsTile = 128;
constexpr unsigned long long kAggregate = 1, kInclusive = 2;   // status word = value << 2 | flag; 0 = not yet published

struct PointsParams {
  FuseParams f;                    // first member: the filter's fields sit at the offsets geo_fuse_kernel reads them from
  double eref_inv[12];             // inv(E_ref) rows 0-2
  const float* image;              // [H,W,3] fp32 in [0,1]
  float* xyz;                      // [capacity,3]
  uint8_t* rgb;                    // [capacity,3]
  long long capacity;
  long long* total;                // in: points before this view; out (last tile): points after it
  unsigned int* ticket;            // workspace word 0
  unsigned long long* status;      // workspace words 1..n_tiles
  int tiles_per_row;
  unsigned int n_tiles;
};
static_assert(sizeof(PointsParams) <= 4096, "PointsParams must stay a small kernel parameter block");

__host__ __device__ inline long long points_tiles(int H, int W) { return (long long)H * ((W + kPointsTile - 1) / kPointsTile); }

__device__ __forceinline__ void publish(unsigned long long* word, unsigned long long flag, long long value) {
  cuda::atomic_ref<unsigned long long, cuda::thread_scope_device>(*word).store(((unsigned long long)value << 2) | flag,
                                                                               cuda::memory_order_release);
}

// Exclusive prefix of tile t (t >= 1), computed by one full warp: each round reads the 32 words before the window's
// end, lane l the word of tile j - l, waiting until it is published, and sums them up to the nearest inclusive one.
// The polls are relaxed and one acquire fence follows the last round: a fence per round cost 13 % of the kernel's time
// (245 vs 214 us at 1152x1600 on a B200), and wider rounds (4 or 8 words per lane) were slower still.
__device__ long long look_back(unsigned long long* status, unsigned int t, int lane) {
  long long sum = 0;
  for (long long j = (long long)t - 1;; j -= 32) {
    const long long k = j - lane;
    unsigned long long s = kInclusive;   // before tile 0: never summed, tile 0 itself is inclusive and nearer
    if (k >= 0) {
      cuda::atomic_ref<unsigned long long, cuda::thread_scope_device> w(status[k]);
      do s = w.load(cuda::memory_order_relaxed); while (s == 0);
    }
    const unsigned inc = __ballot_sync(0xffffffffu, (s & 3) == kInclusive);
    const int stop = inc ? __ffs(inc) - 1 : 31;
    long long v = lane <= stop ? (long long)(s >> 2) : 0;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    sum += v;
    if (inc) {
      cuda::atomic_thread_fence(cuda::memory_order_acquire, cuda::thread_scope_device);
      return sum;
    }
  }
}

// 8 CTAs per SM, as geo_fuse_kernel runs (62 registers, no spills; 72 registers and 7 CTAs without the bound).
__global__ void __launch_bounds__(kPointsTile, 8) geo_points_kernel(const __grid_constant__ PointsParams Q) {
  const FuseParams& P = Q.f;
  __shared__ unsigned int s_tile;
  __shared__ int s_count[kPointsTile / 32];
  __shared__ long long s_base;
  if (threadIdx.x == 0) s_tile = atomicAdd(Q.ticket, 1u);
  __syncthreads();
  const unsigned int t = s_tile;
  const int y = t / Q.tiles_per_row, x = (t % Q.tiles_per_row) * kPointsTile + threadIdx.x;
  const long long pix = (long long)y * P.W + x;
  bool keep = false;
  float wx = 0.f, wy = 0.f, wz = 0.f;
  if (x < P.W) {
    const FusePixel r = fuse_pixel(P, x, y, pix);
    keep = r.photo && r.geo;
    if (keep) {   // inv(E) [inv(K) [x,y,1] d; 1] in float64 (filter/dypcd.py:294-298), d the averaged depth
      const double d = (double)r.depth_avg, px = (double)x * d, py = (double)y * d;
      const double* Ki = P.kref_inv;
      const double cx = Ki[0] * px + Ki[1] * py + Ki[2] * d, cy = Ki[3] * px + Ki[4] * py + Ki[5] * d,
                   cz = Ki[6] * px + Ki[7] * py + Ki[8] * d;
      const double* Ei = Q.eref_inv;
      wx = (float)(Ei[0] * cx + Ei[1] * cy + Ei[2] * cz + Ei[3]);
      wy = (float)(Ei[4] * cx + Ei[5] * cy + Ei[6] * cz + Ei[7]);
      wz = (float)(Ei[8] * cx + Ei[9] * cy + Ei[10] * cz + Ei[11]);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ballot = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) s_count[warp] = __popc(ballot);
  __syncthreads();
  if (warp == 0) {
    long long agg = 0;
#pragma unroll
    for (int i = 0; i < kPointsTile / 32; ++i) agg += s_count[i];
    long long excl = 0;
    if (t != 0) {
      if (lane == 0) publish(Q.status + t, kAggregate, agg);
      excl = look_back(Q.status, t, lane);
    }
    if (lane == 0) {
      // Only tile 0 reads the running total and only the last tile writes it.  The release / acquire chain of
      // inclusive prefixes from tile 0 to the last tile orders the read before the write.
      if (t == 0) excl = *Q.total;
      publish(Q.status + t, kInclusive, excl + agg);
      if (t == Q.n_tiles - 1) *Q.total = excl + agg;
      s_base = excl;
    }
  }
  __syncthreads();
  if (keep) {
    long long i = s_base + __popc(ballot & ((1u << lane) - 1u));
    for (int w = 0; w < warp; ++w) i += s_count[w];
    if (i < Q.capacity) {   // past the capacity only the total counts the point
      const float* c = Q.image + pix * 3;
      Q.xyz[i * 3] = wx; Q.xyz[i * 3 + 1] = wy; Q.xyz[i * 3 + 2] = wz;
      // (img * 255).to(torch.uint8): float32 product, truncated
      Q.rgb[i * 3] = (uint8_t)__float2uint_rz(__fmul_rn(__ldg(c), 255.f));
      Q.rgb[i * 3 + 1] = (uint8_t)__float2uint_rz(__fmul_rn(__ldg(c + 1), 255.f));
      Q.rgb[i * 3 + 2] = (uint8_t)__float2uint_rz(__fmul_rn(__ldg(c + 2), 255.f));
    }
  }
}

// Checks the filter's inputs and fills everything of P but its outputs (host only: no CUDA call).
static int fill_filter_params(FuseParams& P, const char* who, const float* depth_ref, const float* conf1, const float* conf2,
                              const float* conf3, const float* const* depth_src, const double* cams, int n_src, int H, int W,
                              float conf_thr1, float conf_thr2, float conf_thr3, double dist_base, double rel_diff_base) {
  DAMVS_REQUIRE(depth_ref && conf1 && conf2 && conf3 && depth_src && cams, "%s: null pointer", who);
  DAMVS_REQUIRE(n_src >= 1 && n_src <= kMaxFuseSrc, "%s: n_src=%d outside [1,%d]", who, n_src, kMaxFuseSrc);
  DAMVS_REQUIRE(H > 0 && H <= 65535 && W > 0, "%s: bad shape", who);
  P.depth_ref = depth_ref; P.conf[0] = conf1; P.conf[1] = conf2; P.conf[2] = conf3;
  // cams: [K_ref 9][inv(K_ref) 9] then per source view 42 doubles (see FuseParams)
  for (int i = 0; i < 9; ++i) { P.kref[i] = cams[i]; P.kref_inv[i] = cams[9 + i]; }
  for (int v = 0; v < n_src; ++v) {
    DAMVS_REQUIRE(depth_src[v], "%s: depth_src[%d] is null", who, v);
    P.depth_src[v] = depth_src[v];
    for (int i = 0; i < 42; ++i) P.cam[v][i] = cams[18 + v * 42 + i];
  }
  P.conf_thr[0] = conf_thr1; P.conf_thr[1] = conf_thr2; P.conf_thr[2] = conf_thr3;
  P.dist_base = dist_base; P.rel_diff_base = rel_diff_base;
  P.n_src = n_src; P.H = H; P.W = W;
  return DAMVS_OK;
}

}  // namespace damvs

using namespace damvs;

extern "C" int damvs_geo_consistency_fuse(const float* depth_ref, const float* conf1, const float* conf2, const float* conf3,
                                          const float* const* depth_src, const double* cams, int n_src, int H, int W,
                                          float conf_thr1, float conf_thr2, float conf_thr3, double dist_base, double rel_diff_base,
                                          float* depth_avg, uint8_t* photo_mask, uint8_t* geo_mask, uint8_t* final_mask, void* stream) {
  DAMVS_REQUIRE(depth_avg && photo_mask && geo_mask && final_mask, "geo_consistency_fuse: null pointer");
  FuseParams P{};
  const int rc = fill_filter_params(P, "geo_consistency_fuse", depth_ref, conf1, conf2, conf3, depth_src, cams, n_src, H, W,
                                    conf_thr1, conf_thr2, conf_thr3, dist_base, rel_diff_base);
  if (rc != DAMVS_OK) return rc;
  P.depth_avg = depth_avg; P.photo_mask = photo_mask; P.geo_mask = geo_mask; P.final_mask = final_mask;
  dim3 grid((W + 127) / 128, H);
  geo_fuse_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(P);
  DAMVS_LAUNCH_OK("geo_fuse kernel");
  return DAMVS_OK;
}

extern "C" size_t damvs_geo_consistency_points_workspace_bytes(int H, int W) {
  if (H <= 0 || W <= 0) return 0;
  return sizeof(unsigned long long) * (1 + (size_t)points_tiles(H, W));
}

extern "C" int damvs_geo_consistency_points(const float* depth_ref, const float* conf1, const float* conf2, const float* conf3,
                                            const float* const* depth_src, const double* cams, const double* ref_world_from_cam,
                                            int n_src, int H, int W, float conf_thr1, float conf_thr2, float conf_thr3,
                                            double dist_base, double rel_diff_base, const float* image, long long capacity,
                                            float* xyz, uint8_t* rgb, long long* total, void* workspace, void* stream) {
  DAMVS_REQUIRE(ref_world_from_cam && image && xyz && rgb && total && workspace, "geo_consistency_points: null pointer");
  DAMVS_REQUIRE(capacity >= 0, "geo_consistency_points: capacity=%lld is negative", capacity);
  DAMVS_REQUIRE(((uintptr_t)total & 7) == 0 && ((uintptr_t)workspace & 7) == 0,
                "geo_consistency_points: total and workspace must be 8-byte aligned");
  PointsParams Q{};
  const int rc = fill_filter_params(Q.f, "geo_consistency_points", depth_ref, conf1, conf2, conf3, depth_src, cams, n_src, H,
                                    W, conf_thr1, conf_thr2, conf_thr3, dist_base, rel_diff_base);
  if (rc != DAMVS_OK) return rc;
  const long long n_tiles = points_tiles(H, W);
  DAMVS_REQUIRE(n_tiles <= 0x7fffffffLL, "geo_consistency_points: %d x %d has too many tiles", H, W);
  for (int i = 0; i < 12; ++i) Q.eref_inv[i] = ref_world_from_cam[i];
  Q.image = image; Q.xyz = xyz; Q.rgb = rgb; Q.capacity = capacity; Q.total = total;
  Q.ticket = static_cast<unsigned int*>(workspace);
  Q.status = static_cast<unsigned long long*>(workspace) + 1;
  Q.tiles_per_row = (W + kPointsTile - 1) / kPointsTile;
  Q.n_tiles = (unsigned int)n_tiles;
  geo_points_kernel<<<(unsigned int)n_tiles, kPointsTile, 0, (cudaStream_t)stream>>>(Q);
  DAMVS_LAUNCH_OK("geo_points kernel");
  return DAMVS_OK;
}
