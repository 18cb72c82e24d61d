// color_kernels.cuh — inputs of the colour path (SURVEY §8 f3): what the reference computes
// between a detected cone and the classifier network.
//
//   cone_box_mask_kernel     get_reconstructed_cone (src/cone_detection.cpp:222-238) for up to
//                            64 cone centres in ONE pass over the raw cloud: per point a 64-bit
//                            set of matching boxes, per (centre, 32-point row) a ballot word
//   cone_box_scan_kernel     exclusive scan of the per-(centre, tile) counts -> crop offsets
//   cone_box_gather_kernel   order-preserving gather of the matches into packed crops
//   cone_raster_kernel       ColorClassifier.to_image (scripts/color_classifier_server.py:
//                            130-156): 15x12 range image of a crop, one CTA per cone
//
// The reference walks the whole cloud once per cone on the host and ships each crop through a
// ROS service; here the cloud already sits in HBM from the detection pass and only 180 bytes
// per cone travel back.
//
// Crops from the ground node's message (CP_COLOR_CLOUD_GROUNDLESS after a run with ground removal).  In the
// reference's default launch the detector crops from the groundless_cloud message: the points the ground filter
// keeps, in input order, then N - G zero points (src/ground_removal.cpp:79).  The mask kernels keep a point that lies
// in a box only if ground_node_keeps() (evaluated for those points alone), and a box that contains (0, 0) gets the
// N - G zero points after its kept points: counted with the crop offsets, written by the gather kernels.
//
// Exactness.  The box test is the reference's double-precision comparison folded into four
// fp32 bounds by box_bounds (largest / smallest float on the right side of each double bound),
// so the crops are bit-exact.  The raster evaluates the numpy formulas in fp64; the only
// operation that is not correctly rounded on the device is atan2 (<= 2 ulp), which matters
// only if a pixel coordinate lands within a guard band of a rounding boundary (x.5): such a
// cone is flagged CP_CONE_AMBIGUOUS instead of being silently different.
#pragma once
#include "cluster_kernels.cuh"
#include "stream_kernels.cuh"

namespace cp {

constexpr int kConeChunk = 64;  // centres per launch: one bit each in the per-point match set
constexpr int kImgRows = 15, kImgCols = 12, kImgPix = kImgRows * kImgCols;
constexpr u32 kConeEmpty = 1u, kConeBadIndex = 2u, kConeBadIntensity = 4u, kConeAmbiguous = 8u;

struct ConeBoxes {
  u32 n;
  float xlo[kConeChunk], xhi[kConeChunk], ylo[kConeChunk], yhi[kConeChunk];
};

// The ground node's verdict on one point (src/ground_removal.cpp:70-77) as keep_point reaches it: non-finite points
// are dropped, the sector is sector_of's, and the threshold is derived from the frame's sector minima
// (low_key[kNSect], ordered keys) as ground_thresholds_kernel derives it.
__device__ __forceinline__ bool ground_node_keeps(const float4& p, const u32* __restrict__ low_key) {
  if (!finite3(p.x, p.y, p.z)) return false;
  bool ok;
  const float a = atan2_approx(p.y, p.x, ok);
  const int s = sector_of(p.x, p.y, a, ok);
  return !(p.z < __double2float_ru((double)ord2f(__ldg(&low_key[s])) + 0.1));
}

// The zero points the ground node pads frame f's message with: N_f - G_f from the run's cp_frame_counters
// (fc[8 f] = N, fc[8 f + 1] = G); none without a groundless cloud (fc NULL).
__device__ __forceinline__ u32 ground_pad(const u32* __restrict__ fc, u32 f) {
  return fc ? fc[(size_t)f * 8] - fc[(size_t)f * 8 + 1] : 0u;
}

// mask[k][row] = ballot of "point row*32+lane lies in box k"; tile_count[k][tile] = matches of box k
// in the 2048-point tile.  Both start from zero (only non-empty rows are written).
template <int MODE>
__global__ void __launch_bounds__(kStreamThreads) cone_box_mask_kernel(
    const uint8_t* __restrict__ in, Layout L, u64 first_point, u32 n_points, const __grid_constant__ ConeBoxes B,
    const u32* __restrict__ low_key, u32 n_rows, u32 n_tiles, u32* __restrict__ mask, u32* __restrict__ tile_count) {
  // one 32-point row per warp (a single frame is small: many short CTAs beat 64 long ones)
  const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const u32 row = blockIdx.x * kStreamWarps + warp;
  if (row >= n_rows) return;
  const u32 tile = row / kTileWords;
  const u32 idx = row * 32 + lane;
  const bool valid = idx < n_points;
  float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) p = load_point<MODE>(in, first_point + idx, L);
  u32 m0 = 0, m1 = 0;
  for (u32 k = 0; k < B.n; ++k) {
    // NaN coordinates fail every comparison, like the reference's double comparisons
    const bool inside = valid && p.x >= B.xlo[k] && p.x <= B.xhi[k] && p.y >= B.ylo[k] && p.y <= B.yhi[k];
    if (k < 32) m0 |= (u32)inside << k;
    else m1 |= (u32)inside << (k - 32);
  }
  // groundless cloud (low_key = the frame's sector minima): only points inside some box need the ground verdict
  if (low_key && (m0 | m1) && !ground_node_keeps(p, low_key)) m0 = m1 = 0u;
  u32 any0 = __reduce_or_sync(0xFFFFFFFFu, m0), any1 = __reduce_or_sync(0xFFFFFFFFu, m1);
  while (any0 | any1) {
    const bool hi = any0 == 0;
    const u32 bit = hi ? __ffs(any1) - 1 : __ffs(any0) - 1;
    const u32 b = __ballot_sync(0xFFFFFFFFu, ((hi ? m1 : m0) >> bit) & 1u);
    const u32 k = bit + (hi ? 32u : 0u);
    if (lane == 0) {
      mask[(size_t)k * n_rows + row] = b;
      atomicAdd(&tile_count[(size_t)k * n_tiles + tile], (u32)__popc(b));
    }
    if (hi) any1 &= any1 - 1;
    else any0 &= any0 - 1;
  }
}

// One CTA.  Warp w scans the tile counts of centres w, w+32 of this chunk; thread 0 then chains the
// chunk totals onto crop_off (crop_off[k0] was written by the previous chunk, 0 for the first).  Bit k of `origin`:
// box k contains (0, 0) and its crop ends with the frame's ground_pad(fc, frame) zero points.
__global__ void __launch_bounds__(1024) cone_box_scan_kernel(u32 n_centers, u32 k0, u32 n_tiles, u64 origin,
                                                             const u32* __restrict__ fc, u32 frame,
                                                             const u32* __restrict__ tile_count,
                                                             u32* __restrict__ tile_excl, u32* __restrict__ crop_off) {
  __shared__ u32 total[kConeChunk];
  const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (u32 k = warp; k < n_centers; k += 32) {
    u32 carry = 0;
    for (u32 base = 0; base < n_tiles; base += 32) {
      const u32 t = base + lane;
      const u32 c = t < n_tiles ? tile_count[(size_t)k * n_tiles + t] : 0u;
      u32 incl = c;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const u32 o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if ((int)lane >= d) incl += o;
      }
      if (t < n_tiles) tile_excl[(size_t)k * n_tiles + t] = carry + incl - c;
      carry += __shfl_sync(0xFFFFFFFFu, incl, 31);
    }
    if (lane == 0) total[k] = carry;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const u32 pad = origin ? ground_pad(fc, frame) : 0u;
    u64 run = crop_off[k0];
    for (u32 k = 0; k < n_centers; ++k) {
      run += total[k] + (((origin >> k) & 1u) ? pad : 0u);
      crop_off[k0 + k + 1] = run > 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)run;  // saturates: the host reports capacity
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(kStreamThreads) cone_box_gather_kernel(
    const uint8_t* __restrict__ in, Layout L, u64 first_point, u32 n_centers, u32 k0, u32 n_rows, u32 n_tiles,
    u64 origin, const u32* __restrict__ fc, u32 frame, const u32* __restrict__ mask,
    const u32* __restrict__ tile_count, const u32* __restrict__ tile_excl, const u32* __restrict__ crop_off, u32 cap,
    float4* __restrict__ crop_pts) {
  const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const u32 tile = blockIdx.x;
  for (u32 k = 0; k < n_centers; ++k) {
    if (tile_count[(size_t)k * n_tiles + tile] == 0) continue;  // uniform over the CTA
    const u32* mrow = mask + (size_t)k * n_rows + (size_t)tile * kTileWords;
    const u32 r0 = tile * kTileWords + lane, r1 = r0 + 32;
    const u32 w0 = r0 < n_rows ? mrow[lane] : 0u, w1 = r1 < n_rows ? mrow[lane + 32] : 0u;
    const u32 c0 = __popc(w0), c1 = __popc(w1);
    u32 s0 = c0, s1 = c1;  // inclusive scans over the 64 rows of the tile
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 a = __shfl_up_sync(0xFFFFFFFFu, s0, d), b = __shfl_up_sync(0xFFFFFFFFu, s1, d);
      if ((int)lane >= d) { s0 += a; s1 += b; }
    }
    s1 += __shfl_sync(0xFFFFFFFFu, s0, 31);
    const u64 base = (u64)crop_off[k0 + k] + tile_excl[(size_t)k * n_tiles + tile];
#pragma unroll
    for (int r = 0; r < kStreamRows; ++r) {
      const u32 rr = warp * kStreamRows + r;  // row inside the tile: warps own consecutive rows
      const u32 word = rr < 32 ? __shfl_sync(0xFFFFFFFFu, w0, rr) : __shfl_sync(0xFFFFFFFFu, w1, rr - 32);
      const u32 excl = rr < 32 ? __shfl_sync(0xFFFFFFFFu, s0 - c0, rr) : __shfl_sync(0xFFFFFFFFu, s1 - c1, rr - 32);
      if ((word >> lane) & 1u) {
        const u64 dst = base + excl + __popc(word & ((1u << lane) - 1u));
        if (dst < cap) {
          const u32 idx = (tile * kTileWords + rr) * 32 + lane;
          crop_pts[dst] = load_point<MODE>(in, first_point + idx, L);
        }
      }
    }
  }
  // the padding of the boxes that contain the origin, after their kept points, spread over all CTAs
  if (origin) {
    const u32 pad = ground_pad(fc, frame);
    for (u32 k = 0; k < n_centers; ++k) {
      if (!((origin >> k) & 1u)) continue;
      const u64 end = crop_off[k0 + k + 1];
      for (u64 d = end - pad + (u64)blockIdx.x * blockDim.x + threadIdx.x; d < end && d < cap;
           d += (u64)gridDim.x * blockDim.x)
        crop_pts[d] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// src/cone_detection.cpp:226-227 as fp32 bounds: `c + hw >= (double)p` <=> p <= largest float <= c + hw, and
// `c - hw <= (double)p` <=> p >= smallest float >= c - hw (every float is exactly representable as a double)
__host__ __device__ inline void box_bounds(float c, double hw, float* lo, float* hi) {
  const double dhi = (double)c + hw, dlo = (double)c - hw;
  float fhi = (float)dhi, flo = (float)dlo;
  if ((double)fhi > dhi) fhi = nextafterf(fhi, -INFINITY);
  if ((double)flo < dlo) flo = nextafterf(flo, INFINITY);
  *lo = flo;  // NaN centres give NaN bounds: nothing matches, like the reference
  *hi = fhi;
}

// src/cone_detection.cpp:276-278, the centroid moved radially by ext: vector_len = euclidan_dist(p.x, p.y, 0) in
// double, narrowed; p.x / len in float; the sum promotes to double.  On the device explicit _rn intrinsics: no FMA
// contraction.  A centroid at the origin gives NaN, as in the reference.
__host__ __device__ inline void extend_center(float x, float y, double ext, float* ex, float* ey) {
#ifdef __CUDA_ARCH__
  const double s = __dadd_rn(__dmul_rn((double)x, (double)x), __dmul_rn((double)y, (double)y));
  const float len = __double2float_rn(__dsqrt_rn(s));
  *ex = __double2float_rn(__dadd_rn((double)x, __dmul_rn((double)__fdiv_rn(x, len), ext)));
  *ey = __double2float_rn(__dadd_rn((double)y, __dmul_rn((double)__fdiv_rn(y, len), ext)));
#else
  const float len = (float)sqrt((double)x * (double)x + (double)y * (double)y);
  *ex = (float)((double)x + (double)(x / len) * ext);
  *ey = (float)((double)y + (double)(y / len) * ext);
#endif
}

// ---- every cluster of a batch run (cp_batch_cone_colors) ---------------------------------
//   batch_box_kernel     extended centre (src/cone_detection.cpp:276-278) + box bounds + frame of each cluster
//                        (+ the ground node's padding count of a box that contains the origin)
//   batch_mark_kernel    one pass over the raw batch: a (cluster, frame row, ballot) triple for every non-empty
//                        32-point row of every box of the row's frame, sort key cluster << row_bits | row
//   batch_scan_kernel    crop offsets (points per cluster) and triple offsets (rows per cluster)
//   (stable radix sort of the triples: cluster-major, rows in cloud order)
//   batch_gather_kernel  one warp per cluster re-reads its matched rows into the packed crops, then the padding
// Scratch is O(K + triples); a triple holds at least one crop point, so the crop capacity bounds both.
// batch ctl words: [0] triples found, [1] live sort-key bits, [2] triples to sort (min(found, capacity))
constexpr u32 kBatchScanThreads = 1024;

__global__ void __launch_bounds__(256) batch_box_kernel(const ClusterRec* __restrict__ cl, const u32* __restrict__ k_off,
                                                        u32 n_frames, u32 K, double ext, double hw, u32 key_bits,
                                                        const u32* __restrict__ fc, float4* __restrict__ box,
                                                        u32* __restrict__ kframe,
                                                        u32* __restrict__ cnt, u32* __restrict__ tcnt, u32* __restrict__ ctl) {
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) {
    ctl[0] = 0u;
    ctl[1] = key_bits;
  }
  if (k >= K) return;
  u32 lo = 0, hi = n_frames;  // last frame f with k_off[f] <= k (empty frames share their offset with the next)
  while (hi - lo > 1) {
    const u32 mid = (lo + hi) >> 1;
    if (k_off[mid] <= k) lo = mid; else hi = mid;
  }
  float ex, ey;
  extend_center(cl[k].x, cl[k].y, ext, &ex, &ey);
  float4 b;
  box_bounds(ex, hw, &b.x, &b.y);
  box_bounds(ey, hw, &b.z, &b.w);
  box[k] = b;
  kframe[k] = lo;
  // a box that contains (0, 0) ends with the ground node's padding (NaN bounds contain nothing)
  const bool origin = b.x <= 0.0f && b.y >= 0.0f && b.z <= 0.0f && b.w >= 0.0f;
  cnt[k] = origin ? ground_pad(fc, lo) : 0u;
  tcnt[k] = 0u;
}

__device__ __forceinline__ u64 frame_first_point(const Geom& g, u32 f) {
  return g.uniform_n ? (u64)f * g.uniform_n : g.frame_off[f];
}

template <int MODE>
__global__ void __launch_bounds__(kStreamThreads) batch_mark_kernel(
    const uint8_t* __restrict__ in, Layout L, const Geom g, const u32* __restrict__ k_off,
    const float4* __restrict__ box, const u32* __restrict__ low_key, u32 row_bits, u32 cap, u64* __restrict__ keys,
    u32* __restrict__ vals,
    u32* __restrict__ cnt, u32* __restrict__ tcnt, u32* __restrict__ ctl) {
  const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (u32 tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x) {
    u32 frame, local0, count;
    u64 first;
    tile_lookup(g, tile, frame, local0, count, first);
    const u32 kb = k_off[frame], ke = k_off[frame + 1];
    if (kb == ke) continue;  // a frame without clusters is never read
    float4 p[kStreamRows];
    bool valid[kStreamRows];
#pragma unroll
    for (int r = 0; r < kStreamRows; ++r) {
      const u32 i = (warp * kStreamRows + r) * 32 + lane;
      valid[r] = i < count;
      p[r] = valid[r] ? load_point<MODE>(in, first + local0 + i, L) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // NaN coordinates fail every comparison, like the reference's double comparisons
    auto inside = [&](int r, const float4& b) {
      return valid[r] && p[r].x >= b.x && p[r].x <= b.y && p[r].y >= b.z && p[r].y <= b.w;
    };
    // bounding rectangle of the warp's points (fminf / fmaxf skip NaN): a box that misses it holds none of them
    float mnx = INFINITY, mxx = -INFINITY, mny = INFINITY, mxy = -INFINITY;
#pragma unroll
    for (int r = 0; r < kStreamRows; ++r)
      if (valid[r]) {
        mnx = fminf(mnx, p[r].x); mxx = fmaxf(mxx, p[r].x);
        mny = fminf(mny, p[r].y); mxy = fmaxf(mxy, p[r].y);
      }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
      mnx = fminf(mnx, __shfl_xor_sync(kFull, mnx, d)); mxx = fmaxf(mxx, __shfl_xor_sync(kFull, mxx, d));
      mny = fminf(mny, __shfl_xor_sync(kFull, mny, d)); mxy = fmaxf(mxy, __shfl_xor_sync(kFull, mxy, d));
    }
    auto misses = [&](const float4& b) { return b.y < mnx || b.x > mxx || b.w < mny || b.z > mxy; };
    if (low_key) {
      // groundless cloud: a point in some box stays only if the ground node keeps it (low_key: the run's sector
      // minima); points in no box are dropped outright, which changes no ballot
      u32 cand = 0;
      for (u32 k = kb; k < ke; ++k) {
        const float4 b = box[k];
        if (misses(b)) continue;
#pragma unroll
        for (int r = 0; r < kStreamRows; ++r) cand |= (u32)inside(r, b) << r;
      }
      if (!__any_sync(kFull, cand)) continue;
#pragma unroll
      for (int r = 0; r < kStreamRows; ++r)
        valid[r] = ((cand >> r) & 1u) && ground_node_keeps(p[r], low_key + (size_t)frame * kSectStride);
    }
    // count the warp's non-empty (box, row) ballots, reserve that many slots with one atomic, then write them
    u32 n = 0;
    for (u32 k = kb; k < ke; ++k) {
      const float4 b = box[k];
      if (misses(b)) continue;  // uniform over the warp
#pragma unroll
      for (int r = 0; r < kStreamRows; ++r) n += __ballot_sync(kFull, inside(r, b)) != 0u;
    }
    if (n == 0) continue;
    u32 slot = 0;
    if (lane == 0) slot = atomicAdd(&ctl[0], n);
    slot = __shfl_sync(kFull, slot, 0);
    const u32 row0 = local0 / 32 + warp * kStreamRows;
    for (u32 k = kb; k < ke; ++k) {
      const float4 b = box[k];
      if (misses(b)) continue;
      u32 pts = 0, rows = 0;
#pragma unroll
      for (int r = 0; r < kStreamRows; ++r) {
        const u32 bal = __ballot_sync(kFull, inside(r, b));
        if (bal) {
          if (lane == 0 && slot < cap) {
            keys[slot] = ((u64)k << row_bits) | (row0 + r);
            vals[slot] = bal;
          }
          ++slot;
          pts += __popc(bal);
          ++rows;
        }
      }
      if (lane == 0 && rows) {
        atomicAdd(&cnt[k], pts);
        atomicAdd(&tcnt[k], rows);
      }
    }
  }
}

// One CTA: exclusive scans of the per-cluster point and row counts (saturating: the host reports capacity).
__global__ void __launch_bounds__(kBatchScanThreads) batch_scan_kernel(u32 K, const u32* __restrict__ cnt,
                                                                       const u32* __restrict__ tcnt,
                                                                       u32* __restrict__ off, u32* __restrict__ toff,
                                                                       u32 cap, u32* __restrict__ ctl) {
  __shared__ u64 wsum[2][kBatchScanThreads / 32];
  const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  u64 carry0 = 0, carry1 = 0;
  for (u32 base = 0; base < K; base += kBatchScanThreads) {
    const u32 k = base + tid;
    const u64 c0 = k < K ? cnt[k] : 0u, c1 = k < K ? tcnt[k] : 0u;
    u64 s0 = c0, s1 = c1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u64 a = __shfl_up_sync(kFull, s0, d), b = __shfl_up_sync(kFull, s1, d);
      if ((int)lane >= d) { s0 += a; s1 += b; }
    }
    if (lane == 31) { wsum[0][warp] = s0; wsum[1][warp] = s1; }
    __syncthreads();
    u64 w0 = 0, w1 = 0, t0 = 0, t1 = 0;
    for (u32 w = 0; w < kBatchScanThreads / 32; ++w) {
      if (w < warp) { w0 += wsum[0][w]; w1 += wsum[1][w]; }
      t0 += wsum[0][w];
      t1 += wsum[1][w];
    }
    if (k < K) {
      const u64 e0 = carry0 + w0 + s0 - c0, e1 = carry1 + w1 + s1 - c1;
      off[k] = e0 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)e0;
      toff[k] = e1 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)e1;
    }
    carry0 += t0;
    carry1 += t1;
    __syncthreads();
  }
  if (tid == 0) {
    off[K] = carry0 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)carry0;
    toff[K] = carry1 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)carry1;
    ctl[2] = min(ctl[0], cap);
  }
}

// One warp per cluster, over its triples in sorted (cloud) order; crops land at off[k] in the layout of
// cone_box_gather_kernel.  Nothing is written past `cap`; when the triples did not fit, nothing is gathered at
// all (the sorted prefix does not line up with the triple offsets) and the host grows the buffers and runs again.
template <int MODE>
__global__ void __launch_bounds__(256) batch_gather_kernel(
    const uint8_t* __restrict__ in, Layout L, const Geom g, u32 K, const u32* __restrict__ kframe,
    const u64* __restrict__ keys, const u32* __restrict__ vals, const u32* __restrict__ toff,
    const u32* __restrict__ off, u32 row_bits, u32 cap, const u32* __restrict__ ctl, float4* __restrict__ crop_pts) {
  if (ctl[0] > cap) return;
  const u32 lane = threadIdx.x & 31;
  const u32 nwarps = gridDim.x * (blockDim.x >> 5);
  const u64 row_mask = (1ull << row_bits) - 1ull;
  for (u32 k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); k < K; k += nwarps) {
    const u32 t0 = toff[k], t1 = min(toff[k + 1], cap);
    const u64 first = frame_first_point(g, kframe[k]);
    u64 dst0 = off[k];
    for (u32 tb = t0; tb < t1; tb += 32) {
      const u32 t = tb + lane;
      const u32 word = t < t1 ? vals[t] : 0u;
      const u32 row = t < t1 ? (u32)(keys[t] & row_mask) : 0u;
      const u32 c = __popc(word);
      u32 incl = c;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const u32 o = __shfl_up_sync(kFull, incl, d);
        if ((int)lane >= d) incl += o;
      }
      const u32 m = min(32u, t1 - tb);
      for (u32 j = 0; j < m; ++j) {
        const u32 wj = __shfl_sync(kFull, word, j), rj = __shfl_sync(kFull, row, j);
        const u32 ej = __shfl_sync(kFull, incl - c, j);
        if ((wj >> lane) & 1u) {
          const u64 dst = dst0 + ej + __popc(wj & ((1u << lane) - 1u));
          if (dst < cap) crop_pts[dst] = load_point<MODE>(in, first + (u64)rj * 32 + lane, L);
        }
      }
      dst0 += __shfl_sync(kFull, incl, 31);
    }
    // the ground node's padding (batch_box_kernel counted it): zero points up to the next crop
    for (u64 d = dst0 + lane; d < off[k + 1] && d < cap; d += 32) crop_pts[d] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// ---- range image ---------------------------------------------------------------------
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int d = 16; d; d >>= 1) v = fmin(v, __shfl_xor_sync(0xFFFFFFFFu, v, d));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int d = 16; d; d >>= 1) v = fmax(v, __shfl_xor_sync(0xFFFFFFFFu, v, d));
  return v;
}

// distance of t from the nearest rounding boundary of np.round (k + 0.5)
__device__ __forceinline__ double half_distance(double t) { return fabs(fabs(t - floor(t)) - 0.5); }

constexpr int kRasterThreads = 128;
constexpr double kRad2Deg = 57.29577951308232;  // 180.0 / np.pi (np.degrees multiplies by this constant)

__device__ __forceinline__ double horiz_deg(float4 p) { return __dmul_rn(atan2((double)p.y, (double)p.x), kRad2Deg); }
__device__ __forceinline__ double vert_deg(float4 p) {
  const double X = p.x, Y = p.y;
  const double s = __dadd_rn(__dmul_rn(X, X), __dmul_rn(Y, Y));  // pow(X, 2.0) + pow(Y, 2.0): numpy squares
  return __dmul_rn(atan2((double)p.z, __dsqrt_rn(s)), kRad2Deg);
}

// grid = cones; crops packed as float4 {x, y, z, intensity}, cone c = [off[c], off[c+1])
__global__ void __launch_bounds__(kRasterThreads) cone_raster_kernel(const float4* __restrict__ pts,
                                                                     const u32* __restrict__ off, u32 cap,
                                                                     uint8_t* __restrict__ images,
                                                                     u32* __restrict__ flags_out) {
  __shared__ double s_min[kRasterThreads / 32], s_max[kRasterThreads / 32];
  __shared__ int s_last[kImgPix];
  __shared__ u32 s_flags;
  const u32 cone = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 b = off[cone], e = min(off[cone + 1], cap);
  const u32 n = e > b ? e - b : 0u;
  for (u32 i = tid; i < kImgPix; i += kRasterThreads) s_last[i] = -1;
  if (tid == 0) s_flags = n ? 0u : kConeEmpty;  // color_classifier_server.py:83-84 skips empty clouds
  __syncthreads();
  u32 flags = 0;
  double hmin = __longlong_as_double(0x7ff0000000000000LL), hmax = -hmin;
  bool same_xy = true;  // every point at the first point's (x, y): a zero horizontal range is then exact
  for (u32 i = tid; i < n; i += kRasterThreads) {
    const float4 p = pts[b + i];
    const double ha = horiz_deg(p), va = vert_deg(p);
    same_xy = same_xy && p.x == pts[b].x && p.y == pts[b].y;
    if (!isfinite(ha) || !isfinite(va)) flags |= kConeBadIndex;
    if (!(p.w >= 0.0f && p.w <= 255.0f)) flags |= kConeBadIntensity;  // interp1d([0, 255], ...) bounds
    hmin = fmin(hmin, ha);
    hmax = fmax(hmax, ha);
  }
  hmin = warp_min(hmin);
  hmax = warp_max(hmax);
  if (lane == 0) { s_min[warp] = hmin; s_max[warp] = hmax; }
  if (flags) atomicOr(&s_flags, flags);
  const int all_same = __syncthreads_and(same_xy);
  hmin = s_min[0]; hmax = s_max[0];
#pragma unroll
  for (int w = 1; w < kRasterThreads / 32; ++w) { hmin = fmin(hmin, s_min[w]); hmax = fmax(hmax, s_max[w]); }
  const bool usable = s_flags == 0;
  __syncthreads();
  if (usable) {
    // slope_horiz = (IMG_COLS - 1) / (max - min + 1e-16)                                   (:148)
    const double slope_h = __ddiv_rn(11.0, __dadd_rn(__dsub_rn(hmax, hmin), 1e-16));
    // a 2-ulp atan2 error moves an angle by < 4e-13 degrees; scaled by the slope it bounds the pixel error
    const double guard_h = 1e-9 + slope_h * 4e-13, guard_v = 1e-9;
    // distinct points whose azimuths collapse to one value here need not collapse in libm
    flags = (hmax == hmin && !all_same) ? kConeAmbiguous : 0u;
    for (u32 i = tid; i < n; i += kRasterThreads) {
      const float4 p = pts[b + i];
      const double ha = horiz_deg(p), va = vert_deg(p);
      // slope_vert * (vert_angles - MIN_V_ANGLE), slope_vert = 15 / (-15 - 15)               (:139)
      const double tv = __dmul_rn(-0.5, __dsub_rn(va, -15.0));
      const double dh = __dsub_rn(ha, hmin);
      const double th = __dmul_rn(slope_h, dh);
      const double v = rint(tv), hh = rint(th);  // np.round: half to even
      if (half_distance(tv) < guard_v) flags |= kConeAmbiguous;
      if (dh != 0.0 && half_distance(th) < guard_h) flags |= kConeAmbiguous;
      if (!(v >= -kImgRows && v <= kImgRows - 1) || !(hh >= -kImgCols && hh <= kImgCols - 1)) {
        flags |= kConeBadIndex;  // numpy raises IndexError
        continue;
      }
      const int row = v < 0 ? (int)v + kImgRows : (int)v;  // negative numpy indices wrap
      const int col = hh < 0 ? (int)hh + kImgCols : (int)hh;
      atomicMax(&s_last[row * kImgCols + col], (int)i);  // repeated pixels: the last point wins
    }
    if (flags) atomicOr(&s_flags, flags);
  }
  __syncthreads();
  const bool draw = (s_flags & ~kConeAmbiguous) == 0;
  for (u32 i = tid; i < kImgPix; i += kRasterThreads) {
    const int src = s_last[i];
    uint8_t val = 0;
    if (draw && src >= 0) val = (uint8_t)(int)pts[b + src].w;  // identity interp1d, uint8 store truncates
    images[(size_t)cone * kImgPix + i] = val;
  }
  if (tid == 0) flags_out[cone] = s_flags;
}

}  // namespace cp
