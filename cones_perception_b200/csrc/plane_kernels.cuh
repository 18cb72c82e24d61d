// plane_kernels.cuh — the plane ground model (cp_set_ground_plane, contract in include/conesgpu.h): a seeded RANSAC
// plane per frame, then the ground node's message of every frame.  PARITY UNPINNED: the reference's ground node is
// the sector model; oracle/plane_oracle.cpp restates this contract and the tests hold the kernels to it bit for bit.
//
//   plane_hyp_kernel      F*H hypotheses: three splitmix64 draws each, loaded through the staged Layout, plane in
//                         double without contraction, NaN when invalid; zeroes the counts
//   plane_score_kernel    one pass over the batch, one CTA per 2048-point tile: the frame's H planes in shared
//                         memory, a warp ballot per (row, hypothesis), lane h % 32 keeps hypothesis h's count in a
//                         register; one global atomic per (CTA, hypothesis): integer sums, so deterministic
//   plane_select_kernel   one warp per frame: the argmax of the frame's counts (ties to the lowest h)
//   plane_count_kernel    per tile: the verdict under the chosen plane, kept points per tile
//   plane_write_kernel    per tile: the tile's place in its frame's message from the counts of the frame's earlier
//                         tiles, survivors in input order, and the tile's share of the padding
//
// Five launches whatever the batch.  The points are read three times (score, count, write): 48 B per point of
// reads and 32 B of message writes.
#pragma once
#include "stream_kernels.cuh"

namespace cp {

constexpr u32 kPlaneMaxH = 256;

struct PlaneK {
  u64 seed;
  u32 H;
  float inlier;     // scoring: |s| <= inlier
  float height;     // verdict: keep iff s >= height
  double cos_tilt;  // cos(max_tilt_deg), computed once on the host
};

struct PlaneBufs {
  float4* hyp;   // [F*H] a, b, c, d (NaN: invalid)
  u32* cnt;      // [F*H] inliers per hypothesis
  float4* sel;   // [F] the chosen plane (NaN: no valid plane)
  u32* info;     // [F][2] inliers of the chosen plane, its hypothesis (0xFFFFFFFF: none)
  u32* tcount;   // [n_tiles] points each tile keeps
  u32* kept;     // [F] G_f
};

__host__ __device__ __forceinline__ u64 splitmix64(u64 x) {
  u64 z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ u32 plane_draw(u64 seed, u32 h, u32 j, u32 n) {
  return (u32)(((splitmix64(seed + 3ull * h + j) >> 32) * (u64)n) >> 32);
}

__device__ __forceinline__ float4 plane_nan4() {
  const float q = __int_as_float(0x7fc00000);
  return make_float4(q, q, q, q);
}

// the plane through three points, in double with every operation rounded on its own (no FMA contraction)
__device__ __forceinline__ float4 plane_from_points(float4 p0, float4 p1, float4 p2, double cos_tilt) {
  if (!finite3(p0.x, p0.y, p0.z) || !finite3(p1.x, p1.y, p1.z) || !finite3(p2.x, p2.y, p2.z)) return plane_nan4();
  const double x0 = p0.x, y0 = p0.y, z0 = p0.z;
  const double ux = __dsub_rn(p1.x, x0), uy = __dsub_rn(p1.y, y0), uz = __dsub_rn(p1.z, z0);
  const double vx = __dsub_rn(p2.x, x0), vy = __dsub_rn(p2.y, y0), vz = __dsub_rn(p2.z, z0);
  double nx = __dsub_rn(__dmul_rn(uy, vz), __dmul_rn(uz, vy));
  double ny = __dsub_rn(__dmul_rn(uz, vx), __dmul_rn(ux, vz));
  double nz = __dsub_rn(__dmul_rn(ux, vy), __dmul_rn(uy, vx));
  const double L = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)), __dmul_rn(nz, nz)));
  if (!(L > 0.0) || isinf(L)) return plane_nan4();
  if (nz < 0.0) {
    nx = -nx;
    ny = -ny;
    nz = -nz;
  }
  if (__ddiv_rn(nz, L) < cos_tilt) return plane_nan4();
  nx = __ddiv_rn(nx, L);
  ny = __ddiv_rn(ny, L);
  nz = __ddiv_rn(nz, L);
  const double d = -__dadd_rn(__dadd_rn(__dmul_rn(nx, x0), __dmul_rn(ny, y0)), __dmul_rn(nz, z0));
  return make_float4(__double2float_rn(nx), __double2float_rn(ny), __double2float_rn(nz), __double2float_rn(d));
}

__device__ __forceinline__ float plane_distance(const float4& pl, const float4& p) {
  return fmaf(pl.z, p.z, fmaf(pl.y, p.y, fmaf(pl.x, p.x, pl.w)));
}

template <int MODE>
__global__ void __launch_bounds__(256) plane_hyp_kernel(const uint8_t* __restrict__ in, Layout L, Geom g, PlaneK k,
                                                        PlaneBufs b) {
  const u32 total = g.n_frames * k.H;
  for (u32 t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    const u32 f = t / k.H, hh = t - f * k.H;
    const u32 n = g.uniform_n ? g.uniform_n : g.frame_n[f];
    const u64 first = g.uniform_n ? (u64)f * g.uniform_n : g.frame_off[f];
    float4 pl = plane_nan4();
    if (n >= 3) {
      const float4 p0 = load_point<MODE>(in, first + plane_draw(k.seed, hh, 0, n), L);
      const float4 p1 = load_point<MODE>(in, first + plane_draw(k.seed, hh, 1, n), L);
      const float4 p2 = load_point<MODE>(in, first + plane_draw(k.seed, hh, 2, n), L);
      pl = plane_from_points(p0, p1, p2, k.cos_tilt);
    }
    b.hyp[t] = pl;
    b.cnt[t] = 0;
  }
}

// one CTA per tile; out-of-range lanes load NaN and count nowhere
template <int MODE>
__global__ void __launch_bounds__(kStreamThreads) plane_score_kernel(const uint8_t* __restrict__ in, Layout L, Geom g,
                                                                     PlaneK k, PlaneBufs b) {
  __shared__ float4 s_pl[kPlaneMaxH];
  __shared__ u32 s_cnt[kPlaneMaxH];
  const int lane = lane_id();
  u32 frame, local0, count;
  u64 first;
  tile_lookup(g, blockIdx.x, frame, local0, count, first);
  for (u32 i = threadIdx.x; i < k.H; i += kStreamThreads) {
    s_pl[i] = b.hyp[(u64)frame * k.H + i];
    s_cnt[i] = 0;
  }
  __syncthreads();
  float4 p[kStreamRows];
  load_tile<MODE>(in, L, first + local0, count, __int_as_float(0x7fc00000), p);
  bool fin[kStreamRows];
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) fin[r] = finite3(p[r].x, p[r].y, p[r].z);
  u32 acc[kPlaneMaxH / 32];
#pragma unroll
  for (int c = 0; c < (int)(kPlaneMaxH / 32); ++c) {
    acc[c] = 0;
    if ((u32)c * 32 >= k.H) continue;
    const u32 nk = min(32u, k.H - (u32)c * 32);
    for (u32 kk = 0; kk < nk; ++kk) {
      const float4 pl = s_pl[c * 32 + kk];
      u32 n = 0;
#pragma unroll
      for (int r = 0; r < kStreamRows; ++r)
        n += __popc(__ballot_sync(kFull, fin[r] && fabsf(plane_distance(pl, p[r])) <= k.inlier));
      if ((u32)lane == kk) acc[c] += n;
    }
  }
#pragma unroll
  for (int c = 0; c < (int)(kPlaneMaxH / 32); ++c)
    if ((u32)c * 32 + lane < k.H && acc[c]) atomicAdd(&s_cnt[c * 32 + lane], acc[c]);
  __syncthreads();
  for (u32 i = threadIdx.x; i < k.H; i += kStreamThreads)
    if (s_cnt[i]) atomicAdd(&b.cnt[(u64)frame * k.H + i], s_cnt[i]);
}

__device__ __forceinline__ bool plane_keep(const float4& pl, const float4& p, float height) {
  if (!finite3(p.x, p.y, p.z)) return false;
  return isnan(pl.x) || plane_distance(pl, p) >= height;
}

// one warp per frame: the argmax of the frame's counts over its valid hypotheses, ties to the lowest h
__global__ void __launch_bounds__(128) plane_select_kernel(u32 n_frames, PlaneK k, PlaneBufs b) {
  const int lane = lane_id();
  const u32 frame = blockIdx.x * 4u + (threadIdx.x >> 5);
  if (frame >= n_frames) return;
  // key: valid, then the count, then the lowest h
  u64 best = 0;
  for (u32 hh = lane; hh < k.H; hh += 32) {
    const u64 i = (u64)frame * k.H + hh;
    if (isnan(b.hyp[i].x)) continue;
    const u64 key = (1ull << 63) | ((u64)b.cnt[i] << 31) | (u64)(kPlaneMaxH - 1 - hh);
    best = key > best ? key : best;
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    const u64 o = __shfl_xor_sync(kFull, best, d);
    best = o > best ? o : best;
  }
  if (lane == 0) {
    const u32 hh = kPlaneMaxH - 1 - (u32)(best & (kPlaneMaxH - 1));
    b.sel[frame] = best ? b.hyp[(u64)frame * k.H + hh] : plane_nan4();
    b.info[2 * frame] = best ? (u32)((best >> 31) & 0xFFFFFFFFull) : 0u;
    b.info[2 * frame + 1] = best ? hh : 0xFFFFFFFFu;
  }
}

// one CTA per tile: the verdict under the frame's chosen plane, and the tile's kept points
template <int MODE>
__global__ void __launch_bounds__(kStreamThreads) plane_count_kernel(const uint8_t* __restrict__ in, Layout L, Geom g,
                                                                     PlaneK k, PlaneBufs b) {
  __shared__ u32 s_w[kStreamWarps];
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  u32 frame, local0, count;
  u64 first;
  tile_lookup(g, blockIdx.x, frame, local0, count, first);
  const float4 pl = b.sel[frame];
  float4 p[kStreamRows];
  load_tile<MODE>(in, L, first + local0, count, __int_as_float(0x7fc00000), p);
  u32 n = 0;
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) n += __popc(__ballot_sync(kFull, plane_keep(pl, p[r], k.height)));
  if (lane == 0) s_w[warp] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    u32 t = 0;
#pragma unroll
    for (int w = 0; w < kStreamWarps; ++w) t += s_w[w];
    b.tcount[blockIdx.x] = t;
  }
}

// one CTA per tile: frame f's message is out32[32 * frame_off[f] ...) in the PCL PointXYZI layout (x, y, z, 1.0f,
// intensity, 0, 0, 0); the padding points (0, 0, 0, 1.0f, 0, ...) fill the slots after the G_f survivors.  ctl
// non-NULL (the ground calls): every row is counted in rows_loaded, as no row is skipped under the plane model.
template <int MODE>
__global__ void __launch_bounds__(kStreamThreads) plane_write_kernel(const uint8_t* __restrict__ in, Layout L, Geom g,
                                                                     PlaneK k, PlaneBufs b, uint8_t* __restrict__ out32,
                                                                     Ctl* ctl) {
  __shared__ u32 s_w[kStreamWarps], s_excl[kStreamWarps];
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  const u32 tile = blockIdx.x;
  u32 frame, local0, count;
  u64 first;
  tile_lookup(g, tile, frame, local0, count, first);
  const u32 t0 = g.uniform_n ? frame * g.tpf : g.frame_tile0[frame];
  // survivors of the frame's earlier tiles
  u32 part = 0;
  for (u32 j = t0 + threadIdx.x; j < tile; j += kStreamThreads) part += b.tcount[j];
  part = __reduce_add_sync(kFull, part);
  if (lane == 0) s_excl[warp] = part;
  const float4 pl = b.sel[frame];
  float4 p[kStreamRows];
  load_tile<MODE>(in, L, first + local0, count, __int_as_float(0x7fc00000), p);
  u32 bal[kStreamRows], wn = 0;
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) {
    bal[r] = __ballot_sync(kFull, plane_keep(pl, p[r], k.height));
    wn += __popc(bal[r]);
  }
  if (lane == 0) s_w[warp] = wn;
  __syncthreads();
  u32 excl = 0, woff = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kStreamWarps; ++w) {
    excl += s_excl[w];
    if (w < warp) woff += s_w[w];
    total += s_w[w];
  }
  u32 pos = excl + woff;
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) {
    if ((bal[r] >> lane) & 1u) {
      float4* dst = reinterpret_cast<float4*>(out32 + (first + pos + __popc(bal[r] & lanemask_lt())) * 32);
      dst[0] = make_float4(p[r].x, p[r].y, p[r].z, 1.0f);
      dst[1] = make_float4(p[r].w, 0.f, 0.f, 0.f);
    }
    pos += __popc(bal[r]);
  }
  // the padding, split as in mask_compact_kernel<*, true>: this tile dropped d points and the frame's earlier tiles
  // local0 - excl; it fills the d slots just before the last local0 - excl of the message
  const u32 frame_n = g.uniform_n ? g.uniform_n : g.frame_n[frame];
  const u32 d = count - total;
  float4* dst = reinterpret_cast<float4*>(out32 + (first + frame_n - (local0 - excl) - d) * 32);
  for (u32 j = threadIdx.x; j < 2 * d; j += kStreamThreads)
    dst[j] = (j & 1u) ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 1.0f);
  if (threadIdx.x == 0) {
    if (local0 + count == frame_n) b.kept[frame] = excl + total;
    const u32 rows = (count + 31u) / 32u;
    if (ctl && rows) atomicAdd(&ctl->rows_loaded, rows);
  }
}

// n_ground_kept of the detector's counters: G_f of the plane ground node (the detector ran without ground removal
// on the messages, so it wrote N_f there)
__global__ void plane_counters_kernel(u32 n_frames, const u32* __restrict__ kept, u32* __restrict__ fc) {
  for (u32 f = blockIdx.x * blockDim.x + threadIdx.x; f < n_frames; f += gridDim.x * blockDim.x) fc[(u64)f * 8 + 1] = kept[f];
}

}  // namespace cp
