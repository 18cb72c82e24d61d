// stream_kernels.cuh — the streaming front end over the raw scan (16 B/point per pass):
//
//   ground_sector_min_kernel   pass 1 of GroundRemover::cloud_handler
//                              (src/ground_removal.cpp:58-68): per-sector lowest z
//   keep_mask_kernel           pass 2 (:70-77) fused with filter_points_position
//                              (src/cone_detection.cpp:189-204): one keep bit per point
//                              (warp ballots) + survivors per tile
//   tile_scan_kernel           exclusive scan of the per-tile counts (decoupled look-back)
//   gather_survivors_kernel    order-preserving compaction of the few survivors + bbox
//
// The two heavy kernels are pure streaming maps with no inter-CTA dependency: coalesced
// 128-bit loads (one float4 per point in the compact layout), shared-memory sector tables.
// They are instruction-light because of two exact prefilters:
//   pass 1: a point can only lower a sector minimum if z < max over sectors of the minima
//           seen so far, so ground returns above that bound never need their sector;
//   pass 2: a point with z < min over sectors of the thresholds is ground in every sector.
// Exactness: every remaining predicate has a cheap fp32 test with a guard band; points in
// a band (a few per 10^5) re-evaluate the reference's double-precision formula.
#pragma once
#include "common.cuh"

namespace cp {

constexpr int kStreamThreads = 256;
constexpr int kStreamWarps = kStreamThreads / 32;
constexpr int kStreamRows = 8;
constexpr int kStreamTile = kStreamThreads * kStreamRows;  // 2048 points
constexpr int kTileWords = kStreamTile / 32;               // 64 keep-mask words per tile

struct Layout {
  u32 step;
  i32 ox, oy, oz, oi;  // byte offsets; oi < 0 => intensity = 0
  u32 mode;            // 0: compact float4 xyzI, 1: 4-byte aligned fields, 2: byte-wise
};

struct Geom {
  u32 n_frames;
  u32 uniform_n;          // > 0: every frame has this many points
  u32 tpf;                // tiles per frame when uniform
  u32 n_tiles;
  const u32* frame_n;     // [F]
  const u64* frame_off;   // [F] first point of the frame (in points)
  const u32* tile_frame;  // [n_tiles] (ragged batches)
  const u32* frame_tile0; // [F] first tile of the frame
};

struct CropK {
  int do_crop;
  float zthr;                // drop iff z < zthr           (== (double)z < level_threshold)
  double smax, smin;         // drop iff s >= smax || s < smin   (s = x^2+y^2+z^2 in double)
  float smax_lo, smax_hi, smin_lo, smin_hi;  // fp32 guard bands around smax / smin
  float f_hi;                // keep iff |atan2f| < f_hi
  float f_lo_guard, f_hi_guard;
};

struct GroundK {
  int do_ground;
  int want_count;   // = do_ground: ground survivors are counted per frame (n_ground_kept); only the two
                    // experimental front ends still read it
  int pad_survives; // the zero points the ground node pads with survive the crop
};

__device__ __forceinline__ void tile_lookup(const Geom& g, u32 tile, u32& frame, u32& local0, u32& count,
                                            u64& first_point) {
  u32 n;
  if (g.uniform_n) {
    frame = tile / g.tpf;
    local0 = (tile - frame * g.tpf) * kStreamTile;
    first_point = (u64)frame * g.uniform_n;
    n = g.uniform_n;
  } else {
    frame = g.tile_frame[tile];
    local0 = (tile - g.frame_tile0[frame]) * kStreamTile;
    first_point = g.frame_off[frame];
    n = g.frame_n[frame];
  }
  count = n - local0 < (u32)kStreamTile ? n - local0 : (u32)kStreamTile;
}

__device__ __forceinline__ float load_f32_bytes(const uint8_t* p) {
  u32 v = (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24);
  return __uint_as_float(v);
}

template <int MODE>
__device__ __forceinline__ float4 load_point(const uint8_t* base, u64 idx, const Layout& L) {
  if (MODE == 0) {
    return ldg_stream(reinterpret_cast<const float4*>(base) + idx);
  } else if (MODE == 1) {
    const uint8_t* p = base + idx * L.step;
    float4 r;
    r.x = __ldg(reinterpret_cast<const float*>(p + L.ox));
    r.y = __ldg(reinterpret_cast<const float*>(p + L.oy));
    r.z = __ldg(reinterpret_cast<const float*>(p + L.oz));
    r.w = L.oi >= 0 ? __ldg(reinterpret_cast<const float*>(p + L.oi)) : 0.0f;
    return r;
  } else {
    const uint8_t* p = base + idx * L.step;
    float4 r;
    r.x = load_f32_bytes(p + L.ox);
    r.y = load_f32_bytes(p + L.oy);
    r.z = load_f32_bytes(p + L.oz);
    r.w = L.oi >= 0 ? load_f32_bytes(p + L.oi) : 0.0f;
    return r;
  }
}

// ---- angle / sector arithmetic --------------------------------------------------------
// The reference's atan2(float, float) is libm's atan2f: up to glibc 2.40 the classic fdlibm single-precision
// routine, which is not correctly rounded (e.g. atan2f(1.7f, -1.7e-8f) is one float below pi/2).  Parity means
// reproducing that routine, so the exact path restates it operation by operation in IEEE fp32 (explicit _rn
// intrinsics: no FMA contraction).  oracle/cones_oracle.cpp holds the same restatement, checked against libm
// exhaustively (atanf) / on 4.8e9 pairs (atan2f).  Only guard-band points ever come here.
__device__ __forceinline__ float fd_poly(float x, float& s1, float& s2) {
  const float z = __fmul_rn(x, x), w = __fmul_rn(z, z);
  float a = __fmul_rn(w, 1.6285819933e-02f);
  a = __fmul_rn(w, __fadd_rn(4.9768779427e-02f, a));
  a = __fmul_rn(w, __fadd_rn(6.6610731184e-02f, a));
  a = __fmul_rn(w, __fadd_rn(9.0908870101e-02f, a));
  a = __fmul_rn(w, __fadd_rn(1.4285714924e-01f, a));
  s1 = __fmul_rn(z, __fadd_rn(3.3333334327e-01f, a));
  float b = __fmul_rn(w, -3.6531571299e-02f);
  b = __fmul_rn(w, __fadd_rn(-5.8335702866e-02f, b));
  b = __fmul_rn(w, __fadd_rn(-7.6918758452e-02f, b));
  b = __fmul_rn(w, __fadd_rn(-1.1111110449e-01f, b));
  s2 = __fmul_rn(w, __fadd_rn(-2.0000000298e-01f, b));
  return x;
}
__device__ __noinline__ float fdlibm_atanf(float x) {
  const u32 hx = __float_as_uint(x), ix = hx & 0x7fffffffu;
  float hi, lo;
  int id;
  if (ix >= 0x4c000000u) {  // |x| >= 2^25
    if (ix > 0x7f800000u) return __fadd_rn(x, x);
    const float r = __fadd_rn(1.5707962513e+00f, 7.5497894159e-08f);
    return (hx >> 31) ? -r : r;
  }
  if (ix < 0x3ee00000u) {  // |x| < 0.4375
    if (ix < 0x31000000u) return x;
    id = -1;
    hi = lo = 0.f;
  } else {
    x = fabsf(x);
    if (ix < 0x3f980000u) {
      if (ix < 0x3f300000u) {
        id = 0; hi = 4.6364760399e-01f; lo = 5.0121582440e-09f;
        x = __fdiv_rn(__fadd_rn(__fmul_rn(2.0f, x), -1.0f), __fadd_rn(2.0f, x));
      } else {
        id = 1; hi = 7.8539812565e-01f; lo = 3.7748947079e-08f;
        x = __fdiv_rn(__fadd_rn(x, -1.0f), __fadd_rn(x, 1.0f));
      }
    } else {
      if (ix < 0x401c0000u) {
        id = 2; hi = 9.8279368877e-01f; lo = 3.4473217170e-08f;
        x = __fdiv_rn(__fadd_rn(x, -1.5f), __fadd_rn(1.0f, __fmul_rn(1.5f, x)));
      } else {
        id = 3; hi = 1.5707962513e+00f; lo = 7.5497894159e-08f;
        x = __fdiv_rn(-1.0f, x);
      }
    }
  }
  float s1, s2;
  fd_poly(x, s1, s2);
  const float xs = __fmul_rn(x, __fadd_rn(s1, s2));
  if (id < 0) return __fsub_rn(x, xs);
  const float r = __fsub_rn(hi, __fsub_rn(__fsub_rn(xs, lo), x));
  return (hx >> 31) ? -r : r;
}
__device__ __noinline__ float atan2_exact(float y, float x) {
  const float tiny = 1.0e-30f, pi_o_4 = 7.8539818525e-01f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f,
              pi_lo = -8.7422776573e-08f;
  const i32 hx = __float_as_int(x), hy = __float_as_int(y);
  const i32 ix = hx & 0x7fffffff, iy = hy & 0x7fffffff;
  if (ix > 0x7f800000 || iy > 0x7f800000) return __fadd_rn(x, y);
  if (hx == 0x3f800000) return fdlibm_atanf(y);
  const int m = ((hy >> 31) & 1) | ((hx >> 30) & 2);
  if (iy == 0) {
    if (m < 2) return y;
    return m == 2 ? __fadd_rn(pi, tiny) : __fsub_rn(-pi, tiny);
  }
  if (ix == 0) return (hy < 0) ? __fsub_rn(-pi_o_2, tiny) : __fadd_rn(pi_o_2, tiny);
  if (ix == 0x7f800000) {
    if (iy == 0x7f800000) {
      const float q3 = __fmul_rn(3.0f, pi_o_4);
      switch (m) {
        case 0: return __fadd_rn(pi_o_4, tiny);
        case 1: return __fsub_rn(-pi_o_4, tiny);
        case 2: return __fadd_rn(q3, tiny);
        default: return __fsub_rn(-q3, tiny);
      }
    }
    switch (m) {
      case 0: return 0.0f;
      case 1: return -0.0f;
      case 2: return __fadd_rn(pi, tiny);
      default: return __fsub_rn(-pi, tiny);
    }
  }
  if (iy == 0x7f800000) return (hy < 0) ? __fsub_rn(-pi_o_2, tiny) : __fadd_rn(pi_o_2, tiny);
  const i32 k = (iy - ix) >> 23;
  float z;
  if (k > 60) z = __fadd_rn(pi_o_2, __fmul_rn(0.5f, pi_lo));
  else if (hx < 0 && k < -60) z = 0.0f;
  else z = fdlibm_atanf(fabsf(__fdiv_rn(y, x)));
  switch (m) {
    case 0: return z;
    case 1: return __uint_as_float(__float_as_uint(z) ^ 0x80000000u);
    case 2: return __fsub_rn(pi, __fsub_rn(z, pi_lo));
    default: return __fsub_rn(__fsub_rn(z, pi_lo), pi);
  }
}
// src/ground_removal.cpp:20 evaluated at survey time: float((360/16) * M_PI / 180)
#define CP_SECTOR_ANGLE 0.38397244f
#define CP_INV_SECTOR_ANGLE 2.6043537f
#define CP_ANGLE_GUARD 1e-5f     // >= 3x the worst-case error of atan2_approx (3e-6 rad)
#define CP_SECTOR_GUARD 4e-5f    // same bound scaled by 1/sector_angle, plus rounding of u

// src/ground_removal.cpp:61-64 given the exact float angle
__device__ __forceinline__ int sector_from_exact(float a) {
  const float ang = (a < 0.0f) ? (float)((double)a + 6.283185307179586) : a;
  return (int)floorf(__fdiv_rn(ang, CP_SECTOR_ANGLE));
}
__device__ __noinline__ int sector_exact(float x, float y) {
  // common exact case first: +x axis (includes the all-zero filler point): atan2 = +-0
  if (y == 0.0f && (x > 0.0f || (x == 0.0f && !signbit(x)))) return 0;
  return sector_from_exact(atan2_exact(y, x));
}

// Approximate atan2 for the fast paths: octant reduction + odd minimax polynomial
// (degree 11, max error 1.74e-6 rad on [0,1]); total error incl. rounding < 3e-6 rad.
// `ok` is false when the inputs are outside the range where that bound holds.
__device__ __forceinline__ float atan2_approx(float y, float x, bool& ok) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  ok = (mx > 1e-30f) & (mx < 1e30f);
  const float t = __fdividef(mn, mx);
  const float s = t * t;
  float p = -0.011719129f;
  p = fmaf(p, s, 0.052647334f);
  p = fmaf(p, s, -0.11642647f);
  p = fmaf(p, s, 0.19354036f);
  p = fmaf(p, s, -0.33262283f);
  p = fmaf(p, s, 0.99997723f);
  float r = p * t;
  r = ay > ax ? 1.57079637f - r : r;
  r = x < 0.0f ? 3.14159274f - r : r;
  return copysignf(r, y);
}

// sector from the approximate angle; exact re-evaluation inside the guard bands
__device__ __forceinline__ int sector_of(float x, float y, float a, bool ok) {
  const float ang = a < 0.0f ? a + 6.2831855f : a;
  const float u = ang * CP_INV_SECTOR_ANGLE;
  const float fl = floorf(u);
  const float fr = u - fl;
  const bool risky = !ok | (fr < CP_SECTOR_GUARD) | (fr > 1.0f - CP_SECTOR_GUARD) | (fabsf(a) < CP_ANGLE_GUARD);
  if (risky) return sector_exact(x, y);
  return (int)fl;
}

__device__ __forceinline__ bool finite3(float x, float y, float z) {
  // 0 * finite = 0; 0 * inf = NaN; 0 * NaN = NaN
  const float t = fmaf(z, 0.0f, fmaf(y, 0.0f, x * 0.0f));
  return t == 0.0f;
}

// ---- pass 1: per-sector minima ----------------------------------------------------------
// prefilter bounds: max of smin over the sectors a quadrant can reach (slot 0: all sectors);
// a point at or above its bound cannot lower any minimum.  Called by the whole CTA.
__device__ __forceinline__ void sector_bounds(const u32* smin, u32* s_bound) {
  const int lane = lane_id();
  if ((threadIdx.x >> 5) == 0) {
    // quadrant q = 1 + (x<0) + 2*(y<0) reaches sectors {0..4}, {4..8}, {12..16}, {8..12}
    const u32 v = lane < kNSect ? smin[lane] : 0u;
    const u32 ball = __reduce_max_sync(kFull, v);
    const u32 b0 = __reduce_max_sync(kFull, lane <= 4 ? v : 0u);
    const u32 b1 = __reduce_max_sync(kFull, (lane >= 4 && lane <= 8) ? v : 0u);
    const u32 b2 = __reduce_max_sync(kFull, (lane >= 12 && lane <= 16) ? v : 0u);
    const u32 b3 = __reduce_max_sync(kFull, (lane >= 8 && lane <= 12) ? v : 0u);
    if (lane == 0) {
      s_bound[0] = ball; s_bound[1] = b0; s_bound[2] = b1; s_bound[3] = b2; s_bound[4] = b3;
    }
  }
  __syncthreads();
}

// one tile of pass 1 against the CTA's shared sector table (src/ground_removal.cpp:58-68)
// the tile's points, warp-contiguous rows; out-of-range lanes get z = pad_z
// `rows`: bit r set = this warp needs its row r (32 consecutive points, 512 B in the compact layout)
template <int MODE>
__device__ __forceinline__ void load_tile(const uint8_t* __restrict__ in, const Layout& L, u64 base, u32 count,
                                          float pad_z, float4 (&p)[kStreamRows], u32 rows = 0xFFu) {
  const u32 wbase = (threadIdx.x >> 5) * (32 * kStreamRows) + lane_id();
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) {
    const u32 i = wbase + r * 32;
    p[r] = ((i < count) && ((rows >> r) & 1u)) ? load_point<MODE>(in, base + i, L)
                                                : make_float4(0.f, 0.f, pad_z, 0.f);
  }
}

// out-of-range lanes must carry z = +inf (key above every bound, skipped by the prefilter)
__device__ __forceinline__ void sector_min_tile(const float4 (&p)[kStreamRows], u32* smin, const u32* s_bound) {
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) {
    const u32 zk = f2ord(p[r].z);
    const float x = p[r].x, y = p[r].y;
    // points on an axis (or with a vanishing product) use the all-sector bound
    const u32 q = (x * y == 0.0f) ? 0u : 1u + (x < 0.0f ? 1u : 0u) + (y < 0.0f ? 2u : 0u);
    if (zk < s_bound[q]) {
      if (finite3(x, y, p[r].z)) {
        bool ok;
        const float a = atan2_approx(y, x, ok);
        const int s = sector_of(x, y, a, ok);
        if (zk < smin[s]) atomicMin(&smin[s], zk);   // src/ground_removal.cpp:65-67
      }
    }
  }
}

// The streaming pass 1 keeps the CTA's shared table but no per-tile barrier: each warp takes its prefilter
// bounds from the table on its own, once per tile.  Other warps may lower entries at any time, so a warp's
// bounds can be stale, but only ever too high: a stale bound lets more points through to the exact
// `zk < smin[s]` test and cannot change a minimum.  On top of the per-point quadrant bound, a row whose lowest
// key is not below the all-sector bound is dropped whole (one redux next to the one rowmax needs anyway).
template <int MODE>
__global__ void __launch_bounds__(kStreamThreads, 4)
ground_sector_min_kernel(const uint8_t* __restrict__ in, Layout L, Geom g, u32* __restrict__ low_key,
                         u32* __restrict__ rowmax) {
  __shared__ u32 smin[kSectStride];
  // contiguous chunk of tiles per CTA so the shared table is flushed once per frame change
  const u32 per = (g.n_tiles + gridDim.x - 1) / gridDim.x;
  const u32 t0 = blockIdx.x * per;
  const u32 t1 = t0 + per < g.n_tiles ? t0 + per : g.n_tiles;
  const int lane = lane_id();
  u32 cur_frame = 0xFFFFFFFFu;
  for (u32 tile = t0; tile < t1; ++tile) {
    u32 frame, local0, count;
    u64 first;
    tile_lookup(g, tile, frame, local0, count, first);
    if (frame != cur_frame) {  // CTA-uniform: every warp walks the same tiles
      __syncthreads();
      if (cur_frame != 0xFFFFFFFFu && threadIdx.x < kNSect)
        atomicMin(&low_key[cur_frame * kSectStride + threadIdx.x], smin[threadIdx.x]);
      // seed from the frame's global table: the default and whatever other CTAs found so far
      if (threadIdx.x < kSectStride)
        smin[threadIdx.x] = threadIdx.x < kNSect ? __ldcg(&low_key[frame * kSectStride + threadIdx.x]) : 0u;
      cur_frame = frame;
      __syncthreads();
    }
    float4 p[kStreamRows];
    load_tile<MODE>(in, L, first + local0, count, __int_as_float(0x7f800000), p);
    // quadrant q = 1 + (x<0) + 2*(y<0) reaches sectors {0..4}, {4..8}, {12..16}, {8..12}
    const u32 v = lane < kNSect ? *(volatile const u32*)&smin[lane] : 0u;
    const u32 ball = __reduce_max_sync(kFull, v);
    const u32 b1 = __reduce_max_sync(kFull, lane <= 4 ? v : 0u);
    const u32 b2 = __reduce_max_sync(kFull, (lane >= 4 && lane <= 8) ? v : 0u);
    const u32 b3 = __reduce_max_sync(kFull, (lane >= 12 && lane <= 16) ? v : 0u);
    const u32 b4 = __reduce_max_sync(kFull, (lane >= 8 && lane <= 12) ? v : 0u);
    u32 mine = 0;
#pragma unroll
    for (int r = 0; r < kStreamRows; ++r) {
      // out-of-range lanes carry z = +inf: a key above every bound
      const u32 zk = f2ord(p[r].z);
      if (__reduce_min_sync(kFull, zk) < ball) {
        const float x = p[r].x, y = p[r].y;
        // points on an axis (or with a vanishing product) use the all-sector bound
        const u32 bq = (x * y == 0.0f) ? ball : (y < 0.0f ? (x < 0.0f ? b4 : b3) : (x < 0.0f ? b2 : b1));
        if (zk < bq && finite3(x, y, p[r].z)) {
          bool ok;
          const float a = atan2_approx(y, x, ok);
          const int s = sector_of(x, y, a, ok);
          if (zk < smin[s]) atomicMin(&smin[s], zk);   // src/ground_removal.cpp:65-67
        }
      }
      // highest z of every 32-point row (as an ordered key): pass 2 skips rows that lie entirely
      // below the lowest ground threshold without reading them
      const u32 m = __reduce_max_sync(kFull, zk);
      if (lane == r) mine = m;
    }
    if (rowmax && lane < kStreamRows) rowmax[(u64)tile * kTileWords + (threadIdx.x >> 5) * kStreamRows + lane] = mine;
  }
  __syncthreads();
  if (cur_frame != 0xFFFFFFFFu && threadIdx.x < kNSect)
    atomicMin(&low_key[cur_frame * kSectStride + threadIdx.x], smin[threadIdx.x]);
}

// ---- pass 2: keep mask ------------------------------------------------------------------
__device__ __forceinline__ bool crop_keep(const CropK& c, float x, float y, float z) {
  if (z < c.zthr) return false;
  const float sf = fmaf(z, z, fmaf(y, y, x * x));
  bool exact = !(sf < 1e30f);
  exact |= (sf > c.smax_lo) & (sf < c.smax_hi);
  exact |= (sf > c.smin_lo) & (sf < c.smin_hi);
  if (exact) {
    // perception_handling::euclidan_dist, src/perception_handling/utils.cpp:32-34
    const double xd = x, yd = y, zd = z;
    double s = __dadd_rn(__dmul_rn(xd, xd), __dmul_rn(yd, yd));
    s = __dadd_rn(s, __dmul_rn(zd, zd));
    return !(s >= c.smax || s < c.smin);
  }
  return !(sf >= c.smax_hi || sf <= c.smin_lo);
}

struct MaskOut {
  u32* mask;        // [n_tiles * 64] keep bits, word (tile, w*8 + r) covers points w*256 + r*32 .. +31
  u32* tile_count;  // [n_tiles] survivors per tile (+1 on a frame's last tile when pad_survives)
  u32* gcount;      // [F] ground survivors (when want_count)
  u32* rows_loaded; // total 32-point rows pass 2 actually read (statistics for the roofline)
};

// per-frame thresholds: :75  p.z < low + 0.1 in double  <=>  z < roundup_to_float((double)low + 0.1).
// Called by the whole CTA; thr[17] and *thr_min live in shared memory.
__device__ __forceinline__ void ground_thresholds(const u32* __restrict__ low_key, u32 frame, float* thr,
                                                  float* thr_min) {
  const int lane = lane_id();
  if ((threadIdx.x >> 5) == 0) {
    float t = __int_as_float(0x7f800000);
    if (lane < kNSect) {
      t = __double2float_ru((double)ord2f(__ldcg(&low_key[frame * kSectStride + lane])) + 0.1);
      thr[lane] = t;
    }
#pragma unroll
    for (int o2 = 16; o2; o2 >>= 1) t = fminf(t, __shfl_xor_sync(kFull, t, o2));
    if (lane == 0) *thr_min = t;
  }
  __syncthreads();
}

// one tile of pass 2: keep bits (src/ground_removal.cpp:70-77 + src/cone_detection.cpp:189-204)
// keep verdicts of one warp's 8 rows (256 consecutive points starting at tile-local index wbase):
// src/ground_removal.cpp:70-77 + src/cone_detection.cpp:189-204.  Returns this lane's mask word
// (lane r < 8 holds the word of row r) and the warp's survivor count.
__device__ __forceinline__ u32 keep_rows(const float4 (&p)[kStreamRows], u32 wbase, u32 count, const CropK& c,
                                         const GroundK& gk, const float* thr, float thr_min, u32& wcount_out,
                                         u32& gkept_out) {
  const int lane = lane_id();
  u32 wcount = 0, gkept = 0, myword = 0;
#pragma unroll
  for (int r = 0; r < kStreamRows; ++r) {
    const u32 i = wbase + r * 32 + lane;
    const float x = p[r].x, y = p[r].y, z = p[r].z;
    bool keep = false;
    // ground prefilter: below the lowest threshold of any sector => ground everywhere
    // (without the per-frame count, points failing the crop need no ground verdict either)
    if ((i < count) && !(z < thr_min) && finite3(x, y, z)) {
      keep = !c.do_crop || crop_keep(c, x, y, z);
      if (keep || gk.want_count) {
        bool ok;
        const float a = atan2_approx(y, x, ok);
        if (keep && c.do_crop) {
          const float aa = fabsf(a);
          if (!ok | (aa > c.f_lo_guard)) {
            if (ok & (aa >= c.f_hi_guard)) keep = false;
            else keep = fabsf(atan2_exact(y, x)) < c.f_hi;  // src/cone_detection.cpp:200-201
          }
        }
        if (gk.do_ground && (keep || gk.want_count)) {
          const int s = sector_of(x, y, a, ok);
          const bool gkeep = !(z < thr[s]);
          if (gkeep) gkept++;
          keep = keep && gkeep;
        }
      }
    }
    const u32 bal = __ballot_sync(kFull, keep);
    wcount += __popc(bal);
    if (lane == r) myword = bal;
  }
  wcount_out = wcount;
  gkept_out = gkept;
  return myword;
}

// out-of-range lanes carry z = -inf (load_tile pad): dropped by `i < count` anyway
__device__ __forceinline__ void keep_mask_tile(const float4 (&p)[kStreamRows], u32 count, const CropK& c,
                                               const GroundK& gk, const float* thr, float thr_min,
                                               u32* __restrict__ mask_words, u32* wtot, u32& gkept_out) {
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  u32 wcount;
  const u32 myword = keep_rows(p, warp * (32 * kStreamRows), count, c, gk, thr, thr_min, wcount, gkept_out);
  if (lane < kStreamRows) mask_words[warp * kStreamRows + lane] = myword;
  if (lane == 0) wtot[warp] = wcount;
}

// tile epilogue: survivors of the tile (+ the pad record on a frame's last tile); whole CTA
__device__ __forceinline__ void keep_mask_finish(const Geom& g, const GroundK& gk, u32 tile, u32 frame, u32 local0,
                                                 u32 count, const u32* wtot, u32 gkept, const MaskOut& o) {
  if (gk.want_count) {
    const u32 gsum = __reduce_add_sync(kFull, gkept);
    if (lane_id() == 0 && gsum) atomicAdd(&o.gcount[frame], gsum);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    u32 total = 0;
#pragma unroll
    for (int w = 0; w < kStreamWarps; ++w) total += wtot[w];
    const bool last_of_frame = (local0 + count) == (g.uniform_n ? g.uniform_n : g.frame_n[frame]);
    o.tile_count[tile] = total + ((gk.pad_survives && last_of_frame) ? 1u : 0u);
  }
  __syncthreads();
}

// one row (32 consecutive points, one per lane): keep verdict of this lane's point, ground filter first
// (src/ground_removal.cpp:70-77), then the crop on what it keeps (src/cone_detection.cpp:189-204).
// gkept counts the ground node's survivors (cp_frame_counters::n_ground_kept).  thr_min / thr_max are the
// lowest / highest threshold of any sector: below thr_min a point is ground everywhere, at or above thr_max it
// is kept everywhere, and only the points in between need their sector (thr_min = thr_max = -inf: no ground
// removal).
__device__ __forceinline__ bool keep_point(const float4& q, bool in_range, const CropK& c, const GroundK& gk,
                                           const float* thr, float thr_min, float thr_max, u32& gkept) {
  const float x = q.x, y = q.y, z = q.z;
  bool keep = false;
  if (in_range && !(z < thr_min) && finite3(x, y, z)) {
    bool ok = false, have_a = false, gkeep = true;
    float a = 0.0f;
    if (gk.do_ground && z < thr_max) {
      a = atan2_approx(y, x, ok);
      have_a = true;
      gkeep = !(z < thr[sector_of(x, y, a, ok)]);
    }
    if (gkeep) {
      gkept++;
      keep = !c.do_crop || crop_keep(c, x, y, z);
      if (keep && c.do_crop) {
        if (!have_a) a = atan2_approx(y, x, ok);
        const float aa = fabsf(a);
        if (!ok | (aa > c.f_lo_guard)) {
          if (ok & (aa >= c.f_hi_guard)) keep = false;
          else keep = fabsf(atan2_exact(y, x)) < c.f_hi;  // src/cone_detection.cpp:200-201
        }
      }
    }
  }
  return keep;
}

// per-frame ground thresholds, once per frame instead of once per tile:
// :75  p.z < low + 0.1 in double  <=>  z < roundup_to_float((double)low + 0.1).
// thr_f[f*32 + s] for the 17 sectors, thr_f[f*32 + 31] = their minimum, thr_f[f*32 + 30] = their maximum.
__global__ void ground_thresholds_kernel(u32 n_frames, const u32* __restrict__ low_key, float* __restrict__ thr_f) {
  const u32 f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_frames) return;
  float mn = __int_as_float(0x7f800000), mx = -__int_as_float(0x7f800000);
  for (int s = 0; s < kNSect; ++s) {
    const float t = __double2float_ru((double)ord2f(low_key[f * kSectStride + s]) + 0.1);
    thr_f[f * kSectStride + s] = t;
    mn = fminf(mn, t);
    mx = fmaxf(mx, t);
  }
  thr_f[f * kSectStride + 31] = mn;
  thr_f[f * kSectStride + 30] = mx;
}

// Pass 2 as a warp-independent streaming map.  A group is 32 rows = 1024 consecutive points
// (half a tile, one 128 B load of row maxima from pass 1); groups are dealt round-robin over all
// warps, which never meet at a block barrier.  Rows whose highest z lies below the lowest ground
// threshold of any sector are ground in every sector — exact, since z < thr_min <= thr[s] — and
// are neither loaded nor evaluated: on a 64-beam scan ~88 % of the rows.  The rows that remain
// are fetched four at a time (independent loads in flight together).  `mask` and `tile_count`
// must be zero before the launch (skipped rows write nothing).
template <int MODE>
__global__ void __launch_bounds__(kStreamThreads, 4)
keep_mask_kernel(const uint8_t* __restrict__ in, Layout L, Geom g, CropK c, GroundK gk,
                 const float* __restrict__ thr_f, const u32* __restrict__ rowmax, MaskOut o, u32 split_log2) {
  constexpr int kBatch = 4;
  const int lane = lane_id();
  const u32 nwarps = gridDim.x * kStreamWarps;
  const u32 gw = blockIdx.x * kStreamWarps + (threadIdx.x >> 5);
  const u32 ngroups = g.n_tiles * 2u;                          // group G = rows [G*32, G*32+32) of the mask
  // a skipped row lies entirely below every threshold: none of its points survives the ground filter, so it
  // contributes nothing to the per-frame ground count either
  const bool skipping = gk.do_ground && rowmax != nullptr;
  u32 nrows = 0;
  // scan order clusters the rows that cannot be skipped (e.g. the beams above the horizon); a
  // contiguous split would leave most warps idle while a few do all the work
  // (the warp slot is rotated by an odd step every round: with a plain stride the same warps would
  // meet the same ring of every frame whenever the warp count is a multiple of the frame's groups)
  // (a batch of a few frames has fewer groups than the GPU has warps: each group is then shared by
  // 2, 4 or 8 warps, one slice of its rows each, so a single frame is not bound by one warp's 32 rows)
  const u32 nvg = ngroups << split_log2;
  const u32 slice_rows = 32u >> split_log2;
  for (u32 round = 0, g0 = 0; g0 < nvg; ++round, g0 += nwarps) {
    const u32 vg = g0 + (gw + round * 37u) % nwarps;
    if (vg >= nvg) continue;
    const u32 grp = vg >> split_log2, sub = vg & ((1u << split_log2) - 1u);
    const u32 slice = split_log2 ? (((1u << slice_rows) - 1u) << (sub * slice_rows)) : 0xFFFFFFFFu;
    const u32 rk = skipping ? rowmax[(u64)grp * 32 + lane] : 0xFFFFFFFFu;   // lane = row within the group
    const u32 tile = grp >> 1;
    u32 frame, local0, count;
    u64 first;
    tile_lookup(g, tile, frame, local0, count, first);
    const float* thr = thr_f + (size_t)frame * kSectStride;
    const float thr_min = gk.do_ground ? __ldg(thr + 31) : -__int_as_float(0x7f800000);
    const float thr_max = gk.do_ground ? __ldg(thr + 30) : -__int_as_float(0x7f800000);
    const u32 half0 = (grp & 1u) * (kStreamTile / 2);          // tile-local index of the group's first point
    if (gk.pad_survives && (grp & 1u) && lane == 0 && sub == 0 &&
        (local0 + count) == (g.uniform_n ? g.uniform_n : g.frame_n[frame]))
      atomicAdd(&o.tile_count[tile], 1u);                      // the record standing for the zero padding
    u32 todo = __ballot_sync(kFull, rk >= f2ord(thr_min)) & slice;  // bit r: row r of the group must be evaluated
    if (todo == 0) continue;
    nrows += __popc(todo);
    const u32 live = todo;
    u32 myword = 0, gcount = 0, gkept = 0;
    if (todo == 0xFFFFFFFFu) {  // (whole groups only: a slice never has all 32 bits)
      // a fully live group (e.g. a ring above the horizon): straight-line, eight rows per round
#pragma unroll 1
      for (u32 b = 0; b < 4; ++b) {
        float4 p[kStreamRows];
#pragma unroll
        for (int r = 0; r < kStreamRows; ++r) {
          const u32 i = half0 + (b * kStreamRows + r) * 32 + lane;
          p[r] = (i < count) ? load_point<MODE>(in, first + local0 + i, L)
                             : make_float4(0.f, 0.f, -__int_as_float(0x7f800000), 0.f);
        }
#pragma unroll
        for (int r = 0; r < kStreamRows; ++r) {
          const u32 i = half0 + (b * kStreamRows + r) * 32 + lane;
          const u32 bal = __ballot_sync(kFull, keep_point(p[r], i < count, c, gk, thr, thr_min, thr_max, gkept));
          gcount += __popc(bal);
          if ((u32)lane == b * kStreamRows + r) myword = bal;
        }
      }
      todo = 0;
    }
    while (todo) {
      // up to four rows per round: all their loads are issued before the first verdict
      float4 p[kBatch];
      u32 rowid[kBatch];
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        rowid[j] = todo ? (u32)__ffs(todo) - 1u : 0xFFFFFFFFu;
        todo &= todo - 1;
        const u32 i = half0 + rowid[j] * 32 + lane;
        p[j] = (rowid[j] != 0xFFFFFFFFu && i < count) ? load_point<MODE>(in, first + local0 + i, L)
                                                       : make_float4(0.f, 0.f, -__int_as_float(0x7f800000), 0.f);
      }
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        if (rowid[j] == 0xFFFFFFFFu) break;
        const u32 i = half0 + rowid[j] * 32 + lane;
        const bool keep = keep_point(p[j], i < count, c, gk, thr, thr_min, thr_max, gkept);
        const u32 bal = __ballot_sync(kFull, keep);
        gcount += __popc(bal);
        if ((u32)lane == rowid[j]) myword = bal;
      }
    }
    if (gcount) {
      if ((live >> lane) & 1u) o.mask[(u64)grp * 32 + lane] = myword;
      if (lane == 0) atomicAdd(&o.tile_count[tile], gcount);
    }
    if (gk.do_ground) {
      const u32 gsum = __reduce_add_sync(kFull, gkept);
      if (lane == 0 && gsum) atomicAdd(&o.gcount[frame], gsum);
    }
  }
  if (lane == 0 && nrows) atomicAdd(o.rows_loaded, nrows);
}

// ---- both passes in ONE persistent kernel (uniform batches with ground removal) ---------
// Work items are handed out by ticket in the order
//     [pass 1 of frame group 0] [pass 2 of group 0] [pass 1 of group 1] [pass 2 of group 1] ...
// A pass-2 item waits until all pass-1 tiles of its frame have published their minima
// (done[frame] == tiles per frame).  It can only wait on items with smaller tickets, which
// running CTAs hold and which never wait themselves, so the kernel cannot deadlock.  A group
// is a few frames (tens of MB), so pass 2 re-reads its points from the 126 MB L2 instead
// of HBM: the scan crosses the HBM interface once.
struct FusedArgs {
  u32 group_tiles;     // tiles per frame group (multiple of tiles per frame)
  u32 n_groups;
  u32* done;           // [F] pass-1 tiles finished per frame (zeroed before the launch)
  u32* ticket;         // zeroed before the launch
};

template <int MODE>
__global__ void __launch_bounds__(kStreamThreads)
front_fused_kernel(const uint8_t* __restrict__ in, Layout L, Geom g, CropK c, GroundK gk, u32* __restrict__ low_key,
                   MaskOut o, FusedArgs fa) {
  __shared__ u32 smin[kSectStride];
  __shared__ u32 sseed[kSectStride];
  __shared__ u32 s_bound[5];
  __shared__ float thr[kSectStride];
  __shared__ float s_thr_min;
  __shared__ u32 wtot[kStreamWarps];
  __shared__ u32 s_ticket;
  const u32 total_items = fa.n_groups * fa.group_tiles * 2u;
  while (true) {
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(fa.ticket, 1u);
    __syncthreads();
    const u32 t = s_ticket;
    if (t >= total_items) break;
    const u32 blk = t / fa.group_tiles;
    const u32 tile = (blk >> 1) * fa.group_tiles + (t - blk * fa.group_tiles);
    if (tile >= g.n_tiles) continue;   // the last group may be partial
    u32 frame, local0, count;
    u64 first;
    tile_lookup(g, tile, frame, local0, count, first);
    float4 p[kStreamRows];
    if ((blk & 1u) == 0) {
      // ---- pass 1 item: the point loads are in flight while the sector table is seeded
      load_tile<MODE>(in, L, first + local0, count, __int_as_float(0x7f800000), p);
      if (threadIdx.x < kSectStride) {
        const u32 v = threadIdx.x < kNSect ? __ldcg(&low_key[frame * kSectStride + threadIdx.x]) : 0u;
        smin[threadIdx.x] = v;
        sseed[threadIdx.x] = v;
      }
      __syncthreads();
      sector_bounds(smin, s_bound);
      sector_min_tile(p, smin, s_bound);
      __syncthreads();
      if (threadIdx.x < kNSect && smin[threadIdx.x] < sseed[threadIdx.x])
        atomicMin(&low_key[frame * kSectStride + threadIdx.x], smin[threadIdx.x]);
      __syncthreads();
      if (threadIdx.x == 0) {
        __threadfence();  // the CTA's minima (ordered before by the barrier) are visible before the count
        atomicAdd(&fa.done[frame], 1u);
      }
    } else {
      // ---- pass 2 item: all pass-1 tiles of this frame must be in; loads first (L2 hits)
      load_tile<MODE>(in, L, first + local0, count, -__int_as_float(0x7f800000), p);
      if (threadIdx.x == 0) {
        while (((volatile u32*)fa.done)[frame] < g.tpf) __nanosleep(64);
        __threadfence();
      }
      __syncthreads();
      ground_thresholds(low_key, frame, thr, &s_thr_min);
      u32 gkept;
      keep_mask_tile(p, count, c, gk, thr, s_thr_min, o.mask + (u64)tile * kTileWords, wtot, gkept);
      keep_mask_finish(g, gk, tile, frame, local0, count, wtot, gkept, o);
    }
  }
}

// ---- exclusive scan of the tile counts ------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanThreads * kScanItems;

__global__ void __launch_bounds__(kScanThreads)
tile_scan_kernel(Geom g, const u32* __restrict__ tile_count, u32* __restrict__ tile_excl,
                 u32* __restrict__ c_off, u64* desc, Ctl* ctl, u32 cap) {
  __shared__ u32 wsum[kScanThreads / 32];
  __shared__ u32 s_tile, s_excl;
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  const u32 stiles = (g.n_tiles + kScanTile - 1) / kScanTile;
  while (true) {
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctl->ticket[0], 1u);
    __syncthreads();
    const u32 st = s_tile;
    if (st >= stiles) break;
    const u32 i0 = st * kScanTile + threadIdx.x * kScanItems;
    u32 v[kScanItems], cnt = 0;
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) {
      v[j] = (i0 + j < g.n_tiles) ? tile_count[i0 + j] : 0u;
      cnt += v[j];
    }
    u32 inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const u32 t = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    u32 woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kScanThreads / 32; ++w) {
      const u32 t = wsum[w];
      if (w < warp) woff += t;
      total += t;
    }
    if (warp == 0) {
      const u32 e = lookback_exclusive(desc, st, total);
      if (lane == 0) s_excl = e;
    }
    __syncthreads();
    u32 run = s_excl + woff + inc - cnt;
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) {
      const u32 t = i0 + j;
      if (t < g.n_tiles) {
        tile_excl[t] = run;
        run += v[j];
        // a frame's last tile publishes the frame's end offset
        u32 frame, nt;
        if (g.uniform_n) {
          frame = t / g.tpf;
          nt = (t + 1 == (frame + 1) * g.tpf);
        } else {
          frame = g.tile_frame[t];
          nt = (t + 1 == g.n_tiles) || (g.tile_frame[t + 1] != frame);
        }
        if (nt) c_off[frame + 1] = run;
        if (t + 1 == g.n_tiles) {
          ctl->n_surv = run < cap ? run : cap;
          if (run > cap) atomicOr(&ctl->error, kErrSurvivors);
        }
      }
    }
    __syncthreads();
  }
}

// ---- ordered gather of the survivors --------------------------------------------------------
struct GatherOut {
  float4* pts;       // [cap] surviving points
  u32* src;          // [cap] frame-local input index
  u32* frame;        // [cap] frame id
  u32 cap;
  u32* bbox_key;     // [F*8] ordered-int min xyz (0..2) / max xyz (4..6)
  uint8_t* out32;    // mask_compact_kernel<*, true>: the ground node's messages, frame f's at frame_off[f] (PCL
                     // 32-byte layout, padding included)
};

// one warp per tile: lane l owns keep words l and l+32 of the tile
template <int MODE>
__global__ void __launch_bounds__(256)
gather_survivors_kernel(const uint8_t* __restrict__ in, Layout L, Geom g, GroundK gk,
                        const u32* __restrict__ mask, const u32* __restrict__ tile_count,
                        const u32* __restrict__ tile_excl, GatherOut o) {
  const int lane = lane_id();
  const u32 warps = (gridDim.x * blockDim.x) >> 5;
  for (u32 tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; tile < g.n_tiles; tile += warps) {
    const u32 tc = tile_count[tile];
    if (tc == 0) continue;
    u32 frame, local0, count;
    u64 first;
    tile_lookup(g, tile, frame, local0, count, first);
    const u32 excl = tile_excl[tile];
    const u32 w0 = mask[(u64)tile * kTileWords + lane], w1 = mask[(u64)tile * kTileWords + 32 + lane];
    const u32 c0 = __popc(w0), c1 = __popc(w1);
    u32 i0 = c0, i1 = c1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 a = __shfl_up_sync(kFull, i0, d), b = __shfl_up_sync(kFull, i1, d);
      if (lane >= d) {
        i0 += a;
        i1 += b;
      }
    }
    const u32 tot0 = __shfl_sync(kFull, i0, 31), tot1 = __shfl_sync(kFull, i1, 31);
    u32 mnx = 0xFFFFFFFFu, mny = 0xFFFFFFFFu, mnz = 0xFFFFFFFFu, mxx = 0, mxy = 0, mxz = 0;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      u32 w = half ? w1 : w0;
      u32 pos = excl + (half ? tot0 + i1 - c1 : i0 - c0);
      const u32 pbase = (half ? 32 + lane : lane) * 32;  // first point of this word within the tile
      while (w) {
        const int b = __ffs(w) - 1;
        w &= w - 1;
        const u32 i = pbase + b;
        const float4 p = load_point<MODE>(in, first + local0 + i, L);
        if (pos < o.cap) {
          o.pts[pos] = p;
          o.src[pos] = local0 + i;
          o.frame[pos] = frame;
        }
        ++pos;
        const u32 kx = f2ord(p.x), ky = f2ord(p.y), kz = f2ord(p.z);
        mnx = min(mnx, kx); mxx = max(mxx, kx);
        mny = min(mny, ky); mxy = max(mxy, ky);
        mnz = min(mnz, kz); mxz = max(mxz, kz);
      }
    }
    const bool last_of_frame = (local0 + count) == (g.uniform_n ? g.uniform_n : g.frame_n[frame]);
    if (gk.pad_survives && last_of_frame && lane == 0) {
      // one record stands for the N-G zero points appended by src/ground_removal.cpp:79;
      // its multiplicity is applied when the voxel mean is taken
      const u32 pos = excl + tot0 + tot1;
      if (pos < o.cap) {
        o.pts[pos] = make_float4(0.f, 0.f, 0.f, 0.f);
        o.src[pos] = 0xFFFFFFFFu;
        o.frame[pos] = frame;
      }
      const u32 kz = f2ord(0.0f);
      mnx = min(mnx, kz); mxx = max(mxx, kz);
      mny = min(mny, kz); mxy = max(mxy, kz);
      mnz = min(mnz, kz); mxz = max(mxz, kz);
    }
    mnx = __reduce_min_sync(kFull, mnx); mny = __reduce_min_sync(kFull, mny);
    mnz = __reduce_min_sync(kFull, mnz); mxx = __reduce_max_sync(kFull, mxx);
    mxy = __reduce_max_sync(kFull, mxy); mxz = __reduce_max_sync(kFull, mxz);
    if (lane == 0) {
      u32* bb = o.bbox_key + frame * 8;
      atomicMin(bb + 0, mnx); atomicMin(bb + 1, mny); atomicMin(bb + 2, mnz);
      atomicMax(bb + 4, mxx); atomicMax(bb + 5, mxy); atomicMax(bb + 6, mxz);
    }
  }
}

// ---- pass 2 + ordered compaction in ONE pass (general back half, ground node) -----------------
// keep_mask_kernel + tile_scan_kernel + gather_survivors_kernel read the scan twice and walk the survivors bit by
// bit; that is the right shape when 1 % of the points survive and the per-frame kernel consumes the mask, and the
// wrong one for the frames that reach the general back half (config 4: 10 % of 2.6 M points survive, no ground
// removal, so no row can be skipped).  Here a CTA takes a 2048-point tile by ticket, judges its points once
// (same keep_point as everywhere else), ranks the survivors with ballots, finds the tile's offset by decoupled
// look-back and stores the survivors in input order, so the result is the one the three kernels produce.
//
// The look-back is deferred by one tile.  Resolved on the spot, it spent half of the kernel spinning (ncu: 39
// polls per look-back window; 209 us for 8 x 2.6 M points, 106 us with the prefixes replayed from a buffer): the
// tiles just before a tile were ticketed microseconds earlier and are in the same phase, so their aggregates are
// not there yet.  Now a tile publishes its aggregate, parks its survivors (compacted, tile order) in shared
// memory, and its CTA goes on to load and judge its next tile; only then does it come back for the parked tile's
// prefix — by then published long ago — and copies the survivors out with coalesced stores.  A tile with more
// survivors than the stash holds (and every tile of the ground node, whose output keeps most points) resolves on
// the spot and stores from the registers the points were loaded into, as before.
constexpr u32 kStashCap = 1024;   // survivors a parked tile may hold (2 x 18 KB per CTA, 4 CTAs per SM)

template <int MODE, bool OUT32>
__global__ void __launch_bounds__(kStreamThreads, 4)
mask_compact_kernel(const uint8_t* __restrict__ in, Layout L, Geom g, CropK c, GroundK gk,
                    const float* __restrict__ thr_f, const u32* __restrict__ rowmax, u64* desc, u32* ticket,
                    GatherOut o, u32* __restrict__ c_off, u32* __restrict__ gcount, Ctl* ctl) {
  constexpr u32 kStash = OUT32 ? 1u : kStashCap;
  __shared__ float4 st_pts[2][kStash];
  __shared__ unsigned short st_idx[2][kStash];
  __shared__ u32 wtot[kStreamWarps];
  __shared__ u32 s_tile, s_excl;
  __shared__ u32 s_bb[8];
  __shared__ float s_thr[kSectStride];
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  const float kInf = __int_as_float(0x7f800000);
  // the parked tile (uniform across the CTA)
  bool parked = false;
  u32 p_tile = 0, p_frame = 0, p_local0 = 0, p_total = 0, p_pad = 0, p_last = 0;
  u32 cur = 0, my_rows = 0;
  while (true) {
    __syncthreads();
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    if (threadIdx.x < 8) s_bb[threadIdx.x] = threadIdx.x < 4 ? 0xFFFFFFFFu : 0u;
    __syncthreads();
    const u32 tile = s_tile;
    const bool valid = tile < g.n_tiles;
    bool park = false;
    u32 frame = 0, local0 = 0, count = 0, total = 0, pad = 0;
    bool last_of_frame = false;
    if (valid) {
      u64 first;
      tile_lookup(g, tile, frame, local0, count, first);
      if (threadIdx.x < kSectStride) s_thr[threadIdx.x] = gk.do_ground ? thr_f[frame * kSectStride + threadIdx.x] : -kInf;
      __syncthreads();
      const float thr_min = s_thr[31], thr_max = s_thr[30];
      // rows lying entirely below every threshold are ground everywhere: never loaded (see keep_mask_kernel)
      u32 rows = 0xFFu;
      if (gk.do_ground && rowmax) {
        const u32 key_min = f2ord(thr_min);
        const u32 rm = lane < kStreamRows ? rowmax[(u64)tile * kTileWords + warp * kStreamRows + lane] : 0u;
        rows = __ballot_sync(kFull, lane < kStreamRows && rm >= key_min) & 0xFFu;
        my_rows += (u32)__popc(rows);
      } else {
        my_rows += (count + 31u) / 32u > (u32)warp * kStreamRows
                       ? min((count + 31u) / 32u - (u32)warp * kStreamRows, (u32)kStreamRows) : 0u;
      }
      float4 p[kStreamRows];
      load_tile<MODE>(in, L, first + local0, count, -kInf, p, rows);
      const u32 wbase = (u32)warp * (32 * kStreamRows);
      u32 bal[kStreamRows], gkept = 0, wcount = 0;
#pragma unroll
      for (int r = 0; r < kStreamRows; ++r) {
        const u32 i = wbase + r * 32 + lane;
        bal[r] = __ballot_sync(kFull, keep_point(p[r], i < count, c, gk, s_thr, thr_min, thr_max, gkept));
        wcount += __popc(bal[r]);
      }
      if (lane == 0) wtot[warp] = wcount;
      if (gk.do_ground) {
        gkept = __reduce_add_sync(kFull, gkept);
        if (lane == 0 && gkept) atomicAdd(&gcount[frame], gkept);
      }
      __syncthreads();
      u32 woff = 0;
#pragma unroll
      for (int w = 0; w < kStreamWarps; ++w) {
        const u32 t = wtot[w];
        if (w < warp) woff += t;
        total += t;
      }
      const u32 frame_n = g.uniform_n ? g.uniform_n : g.frame_n[frame];
      last_of_frame = (local0 + count) == frame_n;
      // one record stands for the N-G zero points appended by src/ground_removal.cpp:79 (see gather_survivors_kernel)
      pad = (!OUT32 && gk.pad_survives && last_of_frame) ? 1u : 0u;
      park = !OUT32 && total <= kStash;
      u32 excl = 0;
      if (park) {
        if (threadIdx.x == 0) lookback_publish(desc, tile, total + pad);
      } else if (OUT32 && local0 == 0) {
        // every frame is its own message: the scan restarts at each frame's first tile, whose prefix is 0 and whose
        // inclusive prefix is published at once, so the look-back of the frame's later tiles stops there
        if (threadIdx.x == 0) {
          desc_store(desc + tile, kStInc | total);
          if (last_of_frame) c_off[frame + 1] = total;
          if (tile + 1 == g.n_tiles) ctl->n_surv = total;
        }
      } else {
        if (warp == 0) {
          const u32 e = lookback_exclusive(desc, tile, total + pad);
          if (lane == 0) s_excl = e;
        }
        __syncthreads();
        excl = s_excl;
        if (threadIdx.x == 0) {
          const u32 run = excl + total + pad;
          if (last_of_frame) c_off[frame + 1] = run;
          if (tile + 1 == g.n_tiles) {
            ctl->n_surv = run < o.cap ? run : o.cap;
            if (run > o.cap) atomicOr(&ctl->error, kErrSurvivors);
          }
        }
      }
      u32 mnx = 0xFFFFFFFFu, mny = 0xFFFFFFFFu, mnz = 0xFFFFFFFFu, mxx = 0, mxy = 0, mxz = 0;
      u32 pos = excl + woff;    // parked: position inside the tile's compacted list
#pragma unroll
      for (int r = 0; r < kStreamRows; ++r) {
        if ((bal[r] >> lane) & 1u) {
          const u32 at = pos + __popc(bal[r] & lanemask_lt());
          if (park) {
            st_pts[cur][at] = p[r];
            st_idx[cur][at] = (unsigned short)(wbase + r * 32 + lane);
          } else if (OUT32) {   // at < N_f: the frame's message holds every survivor
            float4* dst = reinterpret_cast<float4*>(o.out32 + (first + at) * 32);
            dst[0] = make_float4(p[r].x, p[r].y, p[r].z, 1.0f);
            dst[1] = make_float4(p[r].w, 0.f, 0.f, 0.f);
          } else if (at < o.cap) {
            o.pts[at] = p[r];
            o.src[at] = local0 + wbase + r * 32 + lane;
            o.frame[at] = frame;
          }
          const u32 kx = f2ord(p[r].x), ky = f2ord(p[r].y), kz = f2ord(p[r].z);
          mnx = min(mnx, kx); mxx = max(mxx, kx);
          mny = min(mny, ky); mxy = max(mxy, ky);
          mnz = min(mnz, kz); mxz = max(mxz, kz);
        }
        pos += __popc(bal[r]);
      }
      if (OUT32) {
        // the padding points of the message (src/ground_removal.cpp:79, value-initialised PointXYZI), without a
        // second scan: they are all alike, so any split of the frame's tail between its tiles is right.  This tile
        // dropped d = count - total points and the tiles before it in the frame local0 - excl; it fills the d slots
        // just before the last local0 - excl of the message.  Over the frame these tile [P_f + G_f, P_f + N_f).
        const u32 d = count - total;
        float4* dst = reinterpret_cast<float4*>(o.out32 + (first + frame_n - (local0 - excl) - d) * 32);
        for (u32 j = threadIdx.x; j < 2 * d; j += kStreamThreads)
          dst[j] = (j & 1u) ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 1.0f);
      } else {
        if (pad && threadIdx.x == 0) {
          if (!park) {
            const u32 at = excl + total;
            if (at < o.cap) {
              o.pts[at] = make_float4(0.f, 0.f, 0.f, 0.f);
              o.src[at] = 0xFFFFFFFFu;
              o.frame[at] = frame;
            }
          }
          const u32 kz = f2ord(0.0f);
          mnx = min(mnx, kz); mxx = max(mxx, kz);
          mny = min(mny, kz); mxy = max(mxy, kz);
          mnz = min(mnz, kz); mxz = max(mxz, kz);
        }
        mnx = __reduce_min_sync(kFull, mnx); mny = __reduce_min_sync(kFull, mny);
        mnz = __reduce_min_sync(kFull, mnz); mxx = __reduce_max_sync(kFull, mxx);
        mxy = __reduce_max_sync(kFull, mxy); mxz = __reduce_max_sync(kFull, mxz);
        if (lane == 0 && mxx >= mnx) {
          atomicMin(&s_bb[0], mnx); atomicMin(&s_bb[1], mny); atomicMin(&s_bb[2], mnz);
          atomicMax(&s_bb[4], mxx); atomicMax(&s_bb[5], mxy); atomicMax(&s_bb[6], mxz);
        }
        __syncthreads();
        if (threadIdx.x < 8 && (threadIdx.x & 3u) != 3u && s_bb[4] >= s_bb[0]) {
          u32* bb = o.bbox_key + frame * 8;
          if (threadIdx.x < 4) atomicMin(bb + threadIdx.x, s_bb[threadIdx.x]);
          else atomicMax(bb + threadIdx.x, s_bb[threadIdx.x]);
        }
      }
    }
    // ---- the tile parked one round ago: its prefix, then its survivors out of shared memory
    if (!OUT32 && parked) {
      if (warp == 0) {
        const u32 e = lookback_resolve(desc, p_tile, p_total + p_pad);
        if (lane == 0) s_excl = e;
      }
      __syncthreads();   // (also orders this round's stash writes; the parked tile sits in the other buffer)
      const u32 excl = s_excl;
      if (threadIdx.x == 0) {
        const u32 run = excl + p_total + p_pad;
        if (p_last) c_off[p_frame + 1] = run;
        if (p_tile + 1 == g.n_tiles) {
          ctl->n_surv = run < o.cap ? run : o.cap;
          if (run > o.cap) atomicOr(&ctl->error, kErrSurvivors);
        }
        if (p_pad) {
          const u32 at = excl + p_total;
          if (at < o.cap) {
            o.pts[at] = make_float4(0.f, 0.f, 0.f, 0.f);
            o.src[at] = 0xFFFFFFFFu;
            o.frame[at] = p_frame;
          }
        }
      }
      for (u32 i = threadIdx.x; i < p_total; i += kStreamThreads) {
        const u32 at = excl + i;
        if (at < o.cap) {
          o.pts[at] = st_pts[cur ^ 1u][i];
          o.src[at] = p_local0 + st_idx[cur ^ 1u][i];
          o.frame[at] = p_frame;
        }
      }
    }
    parked = park;
    p_tile = tile; p_frame = frame; p_local0 = local0; p_total = total; p_pad = pad; p_last = last_of_frame ? 1u : 0u;
    cur ^= 1u;
    if (!valid) break;
  }
  my_rows = __shfl_sync(kFull, my_rows, 0);
  if (lane == 0 && my_rows) atomicAdd(&ctl->rows_loaded, my_rows);
}

}  // namespace cp
